"""Integrated Gradients, SmoothGrad and the deletion / insertion faithfulness scores of unidefense_b200.explain restated
in numpy / torch.  TEST INFRASTRUCTURE ONLY.

 - F(x) = log p(target | x): log_softmax(cls_out)[target] for two logits; logsigmoid(z) (target 1) or logsigmoid(-z)
   (target 0) for one logit z.
 - Path point k: p_k = b + alpha_k*(x - b) + sigma*eps_k; acc = sum_k w_k * grad F(p_k) in k order.
 - IG (m steps): alpha_k = k/m, trapezoid weights, attr = (x - b)*acc, delta = sum(attr) - (F(x) - F(b)).
 - SmoothGrad (S draws, noise s): alpha_k = 1, sigma = s*(hi - lo), w_k = 1/S, attr = acc.
 - eps_k of element e: normal e & 3 of the Box-Muller pairs of Philox4x32-10((e >> 2, id_lo, id_hi, k),
   (seed_lo, seed_hi ^ NOISE_TAG)).
 - map = sum_c |attr_c|; faithfulness ranks the map descending (ties by pixel index, NaN last) and at j = 0..K
   replaces / restores the pixels of rank < floor(j*HW/K).
csrc/ud_explain.cu computes the IG points and the accumulation in fp32 in exactly the order of path_point and
accumulate below (bit-identical); the noise here is fp64.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.corrupt import _id_words, _seed_key, box_muller, philox4x32_10

NOISE_TAG = 0x534D5448   # "SMTH"


def ig_tables(m):
    """alpha, w (float64) of m-step Integrated Gradients: m + 1 points, trapezoid weights."""
    alpha = np.arange(m + 1, dtype=np.float64) / m
    w = np.full(m + 1, 1.0 / m)
    w[0] = w[-1] = 0.5 / m
    return alpha, w


def smoothgrad_tables(draws):
    return np.ones(draws), np.full(draws, 1.0 / draws)


def objective(logits, target):
    """F per sample in the logits' dtype."""
    if logits.shape[1] == 1:
        z = logits[:, 0]
        return torch.nn.functional.logsigmoid(torch.where(target == 1, z, -z))
    return torch.log_softmax(logits, dim=1).gather(1, target[:, None])[:, 0]


def predicted(logits):
    return (logits[:, 0] > 0).long() if logits.shape[1] == 1 else logits.argmax(dim=1)


def path_point(x, b, alpha, noise=None):
    """b + alpha*(x - b) (+ noise), in the tensors' dtype, in the kernel's operation order; alpha a python float."""
    p = b + alpha * (x - b)
    return p if noise is None else p + noise


def accumulate(acc, w, g):
    return acc + w * g


def normals(P, sample_id, seed, k):
    """eps_k [P] (fp64) of one sample: element e is normal e & 3 of Philox counter (e >> 2, id, k)."""
    q = np.arange((P + 3) // 4, dtype=np.uint64)
    il, ih = _id_words(sample_id)
    a, b, c, d = philox4x32_10((q, il, ih, k), _seed_key(seed, NOISE_TAG))
    z0, z1 = box_muller(a, b)
    z2, z3 = box_muller(c, d)
    return np.stack([z0, z1, z2, z3], 1).reshape(-1)[:P]


def integrated_gradients(f, grad, x, b, m):
    """fp64 IG of a function f(x) -> scalar with gradient grad(x): (attr, delta)."""
    alpha, w = ig_tables(m)
    acc = np.zeros_like(x)
    for a_k, w_k in zip(alpha, w):
        acc = acc + w_k * grad(b + a_k * (x - b))
    attr = (x - b) * acc
    return attr, attr.sum() - (f(x) - f(b))


def rank_desc(amap):
    """rank [..., HW] of the flattened planes through the kernel's radix keys: inverted order-preserving integer image
    of the float, -0 keyed as +0, NaN after every number; a stable sort of the keys."""
    m = np.ascontiguousarray(amap, dtype=np.float32)
    flat = m.reshape(-1, m.shape[-2] * m.shape[-1]) if m.ndim >= 2 else m[None]
    f = np.where(flat == 0, np.float32(0), flat)
    u = f.view(np.uint32).astype(np.uint64)
    key = np.where(u >> 31 == 1, u ^ 0xFFFFFFFF, u ^ 0x80000000)
    key = np.where(np.isnan(flat), 0xFFFFFFFF, 0xFFFFFFFF - key)
    order = np.argsort(key, axis=1, kind="stable")
    rank = np.empty_like(order)
    np.put_along_axis(rank, order, np.arange(order.shape[1])[None].repeat(order.shape[0], 0), axis=1)
    return rank.reshape(m.shape)


def thresholds(K, HW):
    return [j * HW // K for j in range(K + 1)]


def masked(x, b, rank, t, insertion):
    """The deletion (or insertion) input for threshold t: x [N, C, H, W], b of x's shape, rank [N, H, W]."""
    low = (rank < t)[:, None]
    return torch.where(low != insertion, b, x)


def auc(scores):
    """Trapezoid over j/K of scores [N, K+1]."""
    K = scores.shape[1] - 1
    return (scores[:, :-1] + scores[:, 1:]).sum(1) / (2 * K)
