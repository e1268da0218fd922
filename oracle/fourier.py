"""The Fourier-basis perturbation of unidefense_b200.fourier restated in numpy (fp64).  TEST INFRASTRUCTURE ONLY.

 - canonical(u, v): the lexicographically smaller of (u mod H, v mod W) and ((-u) mod H, (-v) mod W).
 - basis: k(h, w) = (((uu*h) mod H)*W + ((vv*w) mod W)*H) mod (H*W); U = a*cos(2 pi k / (H*W)), a = sqrt(1/(H*W)) when
   2uu = 0 (mod H) and 2vv = 0 (mod W), else sqrt(2/(H*W)).  Unit L2 norm, spectrum only at +-(u, v).
 - signs: r_{n,c} = +1 if bit (c & 31) of word (c >> 5) of Philox4x32-10(((uu << 16) | vv, id_lo, id_hi, 0),
   (seed_lo, seed_hi ^ SIGN_TAG)) is 0, else -1.
 - perturb: y = clip(x + s*cos(2 pi k / (H*W)), lo, hi) with s = r * fp32(fp32(eps) * fp32(a)), the kernel's s, and
   the rest in fp64.  csrc/ud_fourier.cu computes t = k/(H*W) and cospif(2t) in fp32.
"""
from __future__ import annotations

import numpy as np

from oracle.corrupt import _id_words, _seed_key, philox4x32_10

SIGN_TAG = 0x464F5552   # "FOUR"


def canonical(u, v, H, W):
    return min((u % H, v % W), ((-u) % H, (-v) % W))


def default_stride(H, W, radius):
    return (min(H, W) // 2) // radius


def grid(H, W, radius, stride=None):
    """-> (u [2R+1], v [R+1], {canonical pair: [(i, j) grid positions]})."""
    s = default_stride(H, W, radius) if stride is None else stride
    u = [a * s for a in range(-radius, radius + 1)]
    v = [b * s for b in range(radius + 1)]
    groups = {}
    for i, uu in enumerate(u):
        for j, vv in enumerate(v):
            groups.setdefault(canonical(uu, vv, H, W), []).append((i, j))
    return u, v, groups


def phase(uu, vv, H, W):
    """k(h, w) [H, W] as int64."""
    h = np.arange(H, dtype=np.int64)[:, None]
    w = np.arange(W, dtype=np.int64)[None, :]
    return (((uu * h) % H) * W + ((vv * w) % W) * H) % (H * W)


def amplitude(uu, vv, H, W):
    return np.sqrt((1.0 if (2 * uu) % H == 0 and (2 * vv) % W == 0 else 2.0) / (H * W))


def basis(u, v, H, W):
    """U_{u,v} [H, W] in fp64, for any signed (u, v)."""
    uu, vv = canonical(u, v, H, W)
    return amplitude(uu, vv, H, W) * np.cos(2 * np.pi * phase(uu, vv, H, W) / (H * W))


def signs(ids, C, uu, vv, seed):
    """r [N, C] (+-1.0) for int sample ids and the canonical (uu, vv)."""
    out = np.empty((len(ids), C))
    key = _seed_key(seed, SIGN_TAG)
    for n, i in enumerate(ids):
        il, ih = _id_words(i)
        words = philox4x32_10(((uu << 16) | vv, il, ih, 0), key)
        for c in range(C):
            out[n, c] = -1.0 if (int(words[c >> 5]) >> (c & 31)) & 1 else 1.0
    return out


def step(uu, vv, H, W, eps, r):
    """s = r * fp32(fp32(eps) * fp32(a)), as the kernel forms it; r [N, C] -> [N, C] float64."""
    m = np.float32(eps) * np.float32(amplitude(uu, vv, H, W))
    return r * np.float64(m)


def perturb(x, uu, vv, eps, ids, seed, lo=-1.0, hi=1.0):
    """y (fp64) = clip(x + s*cos(2 pi k / (H*W)), lo, hi) for x [N, C, H, W] at the canonical (uu, vv)."""
    x = np.asarray(x, dtype=np.float64)
    N, C, H, W = x.shape
    s = step(uu, vv, H, W, eps, signs(ids, C, uu, vv, seed))
    c = np.cos(2 * np.pi * phase(uu, vv, H, W) / (H * W))
    return np.clip(x + s[:, :, None, None] * c, float(np.float32(lo)), float(np.float32(hi)))
