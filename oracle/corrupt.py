"""The image corruptions of unidefense_b200.corrupt restated in numpy.  TEST INFRASTRUCTURE ONLY.

Every corruption maps the input x (fp32 [N, 3, H, W], channels R, G, B, values in [lo, hi]) to 8-bit levels
p = clamp(rint((x - lo)*s), 0, 255) with s = 255/(hi - lo), corrupts the levels, rounds with rint, clamps to [0, 255]
and maps back as lo + p'*(1/s).  csrc/ud_corrupt.cu implements the same definitions:
 - saturation, contrast, block and pixelate here are fp32 statements in the kernel's operation order (no FMA), so the
   kernel is bit-identical to them;
 - noise, blur and jpeg are fp64 definitions.  They also return an "uncertain" mask of the output elements whose value
   a last-bit difference could move: the pre-rounding value lies within UNCERTAIN of a half-integer, or (jpeg) the
   element lies in, or on the one-pixel ring around, a 16x16 MCU holding a DCT coefficient with
   |F/Q - (k + 1/2)| < COEF_UNCERTAIN.  The kernel computes the forward DCT and the quantisation in fp64, so its
   coefficients agree with these to ~1e-12; with a 1e-3 band the MCU rule would cover 2-37 % of the pixels of a
   natural-looking image at q = 90 (a quantisation step of 1-3 leaves many coefficients' fractions spread evenly).
The random corruptions are keyed by a per-sample int64 id and a uint64 seed through Philox4x32-10.
"""
from __future__ import annotations

import numpy as np
from scipy.fft import dctn, idctn

UNCERTAIN = 1e-3
COEF_UNCERTAIN = 1e-9
f32 = np.float32

LEVELS = {
    "saturation": (0.4, 0.3, 0.2, 0.1, 0.0),
    "contrast": (0.85, 0.725, 0.6, 0.475, 0.35),
    "block": (16, 32, 48, 64, 80),
    "noise": (0.001, 0.002, 0.005, 0.01, 0.05),
    "blur": (7, 9, 13, 17, 21),
    "pixelate": (2, 3, 4, 5, 6),
    "jpeg": (90, 70, 50, 30, 10),
}
KINDS = tuple(LEVELS)

BLOCK_TAG = 0x424C4F43   # "BLOC"
NOISE_TAG = 0x4E4F4953   # "NOIS"

# ---- Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11) --------------------------
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: 4 arrays (or ints) of 32-bit words, key: 2.  Returns the 4 output words as uint64 arrays."""
    c = [np.asarray(v, dtype=np.uint64) & _MASK for v in ctr]
    k0, k1 = (np.asarray(v, dtype=np.uint64) & _MASK for v in key)
    for r in range(10):
        p0 = np.uint64(_M0) * c[0]
        p1 = np.uint64(_M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
        k0 = (k0 + np.uint64(_W0)) & _MASK
        k1 = (k1 + np.uint64(_W1)) & _MASK
    return c


def _id_words(i):
    u = int(i) & 0xFFFFFFFFFFFFFFFF
    return u & 0xFFFFFFFF, u >> 32


def _seed_key(seed, tag):
    s = int(seed) & 0xFFFFFFFFFFFFFFFF
    return s & 0xFFFFFFFF, (s >> 32) ^ tag


def box_muller(a, b):
    """Two standard normals from two 32-bit words: u1 = (a + 0.5)*2^-32 in (0, 1), u2 = b*2^-32."""
    u1 = (a.astype(np.float64) + 0.5) * 2.0 ** -32
    u2 = b.astype(np.float64) * 2.0 ** -32
    r = np.sqrt(-2.0 * np.log(u1))
    return r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2)


def block_squares(k, H, W, sample_id, seed):
    """Top-left corners (r, c) of the k 8x8 squares: square j depends on j only, so the squares nest across k."""
    j = np.arange(k, dtype=np.uint64)
    il, ih = _id_words(sample_id)
    u = philox4x32_10((j, il, ih, 0), _seed_key(seed, BLOCK_TAG))
    r = (u[0] * np.uint64(H - 7)) >> np.uint64(32)
    c = (u[1] * np.uint64(W - 7)) >> np.uint64(32)
    return np.stack([r, c], 1).astype(np.int64)


def noise_normals(H, W, sample_id, seed):
    """z0, z1, z2 [H, W]: the normals added to Y, Cb and Cr."""
    n = np.arange(H * W, dtype=np.uint64)
    il, ih = _id_words(sample_id)
    a, b, c, d = philox4x32_10((n, il, ih, 0), _seed_key(seed, NOISE_TAG))
    z0, z1 = box_muller(a, b)
    z2, _ = box_muller(c, d)
    return z0.reshape(H, W), z1.reshape(H, W), z2.reshape(H, W)


# ---- levels ---------------------------------------------------------------------------------------------------------
def scales(lo, hi):
    s = 255.0 / (float(f32(hi)) - float(f32(lo)))
    return f32(s), f32(1.0 / s)


def to_levels(x, lo, hi):
    s, _ = scales(lo, hi)
    return np.clip(np.rint((x.astype(f32) - f32(lo)) * s), f32(0), f32(255)).astype(f32)


def from_levels(p, lo, hi):
    _, inv = scales(lo, hi)
    return (f32(lo) + p.astype(f32) * inv).astype(f32)


def _round(v):
    return np.clip(np.rint(v), 0, 255)


def _near_half(v, band=UNCERTAIN):
    return np.abs(v - np.floor(v) - 0.5) < band


# ---- the four exact kinds (fp32, kernel operation order) ------------------------------------------------------------
def contrast(p, c):
    return _round(p * f32(c)).astype(f32)


def saturation(p, s):
    R, G, B = p[:, 0], p[:, 1], p[:, 2]
    s, h = f32(s), f32(128)
    Y = (f32(0.299) * R + f32(0.587) * G) + f32(0.114) * B
    Cb = ((f32(-0.168736) * R - f32(0.331264) * G) + f32(0.5) * B) + h
    Cr = ((f32(0.5) * R - f32(0.418688) * G) - f32(0.081312) * B) + h
    Cb = h + (Cb - h) * s
    Cr = h + (Cr - h) * s
    R2 = Y + f32(1.402) * (Cr - h)
    G2 = (Y - f32(0.344136) * (Cb - h)) - f32(0.714136) * (Cr - h)
    B2 = Y + f32(1.772) * (Cb - h)
    return _round(np.stack([R2, G2, B2], 1)).astype(f32)


def pixelate(p, f):
    f = int(f)
    N, C, H, W = p.shape
    out = np.empty_like(p)
    for i in range(0, H, f):
        for j in range(0, W, f):
            cell = p[:, :, i:i + f, j:j + f]
            cnt = cell.shape[2] * cell.shape[3]
            s = cell.sum(axis=(2, 3), dtype=np.float64).astype(f32)       # integers <= 255*f*f: exact in fp32
            out[:, :, i:i + f, j:j + f] = _round(s / f32(cnt))[:, :, None, None]
    return out.astype(f32)


def block(p, k, ids, seed):
    N, C, H, W = p.shape
    out = p.copy()
    for n in range(N):
        for r, c in block_squares(int(k), H, W, ids[n], seed):
            out[n, :, r:r + 8, c:c + 8] = 128
    return out


# ---- the fp64 kinds -------------------------------------------------------------------------------------------------
def _ycc(p):
    R, G, B = (p[:, i].astype(np.float64) for i in range(3))
    Y = 0.299 * R + 0.587 * G + 0.114 * B
    Cb = -0.168736 * R - 0.331264 * G + 0.5 * B + 128
    Cr = 0.5 * R - 0.418688 * G - 0.081312 * B + 128
    return Y, Cb, Cr


def _rgb(Y, Cb, Cr):
    return np.stack([Y + 1.402 * (Cr - 128), Y - 0.344136 * (Cb - 128) - 0.714136 * (Cr - 128),
                     Y + 1.772 * (Cb - 128)], 1)


def noise(p, var, ids, seed):
    N, C, H, W = p.shape
    sig = np.sqrt(float(var))
    Y, Cb, Cr = (v / 255.0 for v in _ycc(p))
    for n in range(N):
        z0, z1, z2 = noise_normals(H, W, ids[n], seed)
        Y[n] += sig * z0
        Cb[n] += sig * z1
        Cr[n] += sig * z2
    h = 128 / 255.0
    return 255.0 * np.stack([Y + 1.402 * (Cr - h), Y - 0.344136 * (Cb - h) - 0.714136 * (Cr - h),
                             Y + 1.772 * (Cb - h)], 1)


def blur_weights(k):
    k = int(k)
    r = (k - 1) // 2
    sig = k / 6.0
    i = np.arange(-r, r + 1, dtype=np.float64)
    w = np.exp(-i * i / (2 * sig * sig))
    return w / w.sum()


def reflect101(i, n):
    """OpenCV's BORDER_REFLECT_101 for |overhang| < n: ... c b | a b c ... (the edge is not repeated)."""
    i = np.abs(np.asarray(i))
    return np.where(i >= n, 2 * (n - 1) - i, i)


def blur(p, k):
    N, C, H, W = p.shape
    w = blur_weights(k)
    r = (int(k) - 1) // 2
    v = p.astype(np.float64)
    t = sum(w[i + r] * v[:, :, :, reflect101(np.arange(W) + i, W)] for i in range(-r, r + 1))
    return sum(w[i + r] * t[:, :, reflect101(np.arange(H) + i, H), :] for i in range(-r, r + 1))


# ---- baseline JPEG, 4:2:0 -------------------------------------------------------------------------------------------
LUM = np.array([16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
                14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
                49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99], np.int64).reshape(8, 8)
CHR = np.full((8, 8), 99, np.int64)
CHR[:4, :4] = np.array([17, 18, 24, 47, 18, 21, 26, 66, 24, 26, 56, 99, 47, 66, 99, 99]).reshape(4, 4)


def qtable(T, q):
    """ITU-T T.81 Annex K table T scaled to quality q as libjpeg's jpeg_quality_scaling / jpeg_add_quant_table."""
    q = min(max(int(q), 1), 100)
    S = 5000 // q if q < 50 else 200 - 2 * q
    return np.clip((T * S + 50) // 100, 1, 255)


def _rha(v):
    return np.sign(v) * np.floor(np.abs(v) + 0.5)


def _pad(a, m):
    H, W = a.shape
    return np.pad(a, ((0, -H % m), (0, -W % m)), mode="edge")


def _code(plane, Q):
    """DCT -> quantise -> IDCT per 8x8 block; also the [Hb, Wb] blocks holding a near-tie coefficient."""
    H, W = plane.shape
    b = _pad(plane, 8) - 128.0
    Hp, Wp = b.shape
    b = b.reshape(Hp // 8, 8, Wp // 8, 8).transpose(0, 2, 1, 3)
    F = dctn(b, axes=(2, 3), norm="ortho") / Q
    tie = _near_half(F, COEF_UNCERTAIN).any(axis=(2, 3))
    r = idctn(_rha(F) * Q, axes=(2, 3), norm="ortho").transpose(0, 2, 1, 3).reshape(Hp, Wp) + 128.0
    return r[:H, :W], tie


def _fancy_up(c, H, W):
    """libjpeg's triangle upsampling by 2 per axis: 3/4 of the nearer sample + 1/4 of the next one, edges clamped."""
    def up1(a, n, axis):
        m = a.shape[axis]
        i = np.arange(n)
        near = np.clip(i // 2, 0, m - 1)
        far = np.clip(np.where(i % 2 == 0, i // 2 - 1, i // 2 + 1), 0, m - 1)
        return 0.75 * np.take(a, near, axis=axis) + 0.25 * np.take(a, far, axis=axis)
    return up1(up1(c, H, 0), W, 1)


def _jpeg1(p, q):
    """One image, levels [3, H, W] -> (pre-rounding RGB [3, H, W] fp64, uncertain-MCU mask [H, W])."""
    Y, Cb, Cr = (v[0] for v in _ycc(p[None]))
    H, W = Y.shape

    def down(c):
        c = _pad(c, 2)
        return c.reshape(c.shape[0] // 2, 2, c.shape[1] // 2, 2).mean(axis=(1, 3))

    Yd, ty = _code(Y, qtable(LUM, q))
    Cbd, tb = _code(down(Cb), qtable(CHR, q))
    Crd, tr = _code(down(Cr), qtable(CHR, q))
    Mh, Mw = tb.shape                                   # MCUs: ceil(H/16) x ceil(W/16)
    ty = np.pad(ty, ((0, 2 * Mh - ty.shape[0]), (0, 2 * Mw - ty.shape[1])))
    mcu = ty.reshape(Mh, 2, Mw, 2).any(axis=(1, 3)) | tb | tr
    m = np.zeros((Mh * 16 + 2, Mw * 16 + 2), bool)       # with a one-pixel ring
    for i, j in zip(*np.nonzero(mcu)):
        m[16 * i:16 * i + 18, 16 * j:16 * j + 18] = True
    v = _rgb(Yd[None], _fancy_up(Cbd, H, W)[None], _fancy_up(Crd, H, W)[None])[0]
    return v, m[1:H + 1, 1:W + 1]


def jpeg(p, q):
    out = [_jpeg1(p[n], q) for n in range(p.shape[0])]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])[:, None].repeat(3, 1)


# ---- the whole corruption -------------------------------------------------------------------------------------------
def corrupt(x, kind, param, ids=None, seed=0, lo=-1.0, hi=1.0):
    """x fp32 [N, 3, H, W] (numpy or CPU tensor) -> (y fp32 numpy, uncertain bool mask or None for the exact kinds)."""
    x = np.asarray(x, dtype=f32)
    N = x.shape[0]
    ids = np.arange(N) if ids is None else np.asarray(ids)
    p = to_levels(x, lo, hi)
    unc = None
    if kind == "contrast":
        q = contrast(p, param)
    elif kind == "saturation":
        q = saturation(p, param)
    elif kind == "pixelate":
        q = pixelate(p, param)
    elif kind == "block":
        q = block(p, param, ids, seed)
    else:
        if kind == "noise":
            v, unc = noise(p, param, ids, seed), None
        elif kind == "blur":
            v, unc = blur(p, param), None
        elif kind == "jpeg":
            v, unc = jpeg(p, param)
        else:
            raise ValueError(f"unknown corruption {kind!r}")
        near = _near_half(v)
        unc = near if unc is None else (unc | near)
        q = _round(v).astype(f32)
    return from_levels(q, lo, hi), unc


def test_images(N, H, W, seed=0, lo=-1.0, hi=1.0):
    """Seeded natural-looking test images, fp32 [N, 3, H, W] in [lo, hi]: smooth colour blobs, a diagonal texture, a
    vertical edge and mild sensor noise (not on the 8-bit grid, so the level mapping is exercised too)."""
    g = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W] / max(H, W)
    out = np.empty((N, 3, H, W), f32)
    for n in range(N):
        img = np.zeros((3, H, W))
        for _ in range(12):
            cy, cx, s = g.random(), g.random(), 0.05 + 0.3 * g.random()
            img += g.random(3)[:, None, None] * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * s * s))
        img += 0.15 * np.sin(40 * xx + 25 * yy) * g.random(3)[:, None, None]
        img += (xx > 0.5) * 0.2
        img += 0.03 * g.standard_normal((3, H, W))
        img = (img - img.min()) / (img.max() - img.min())
        out[n] = lo + img * (hi - lo)
    return out
