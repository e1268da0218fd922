"""Closed forms of the input-image gradients of the hot path.  TEST INFRASTRUCTURE ONLY.

The reference differentiates x wherever it enters (model/unidefense.py): the reconstruction losses (rec - x, rfft2(x);
:244-253), the attention error maps (x is resized and enters p - xs and rfft2(p - xs); :126-134, :148), and through
them the guide channels of both dynamic filters (model/modules.py:101-103, :130-132).  Each function below states the
gradient the CUDA kernels compute, in terms of the forward restatements of oracle/recon_path.py; tests/
test_input_grad_oracle.py checks every one against torch autograd of those forwards in fp64, and the forwards are pinned
to the live reference's fixtures (tests/test_oracle_golden.py), so autograd of them stands for the reference's.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import recon_path as O

Tensor = torch.Tensor


def bilinear_align_corners_transpose(g: Tensor, in_size: Sequence[int]) -> Tensor:
    """Adjoint of O.bilinear_align_corners(x -> g.shape[-2:]) for x of spatial size `in_size`
    (upsample_bilinear2d_backward): scatter-add along each axis with the forward's taps."""
    h, w = int(in_size[0]), int(in_size[1])
    H, W = g.shape[-2:]
    y0, y1, ly0, ly1 = O._ac_axis(h, H, g.dtype, g.device)
    x0, x1, lx0, lx1 = O._ac_axis(w, W, g.dtype, g.device)
    tmp = torch.zeros(*g.shape[:-1], w, dtype=g.dtype, device=g.device)
    tmp.index_add_(-1, x0, g * lx0)
    tmp.index_add_(-1, x1, g * lx1)
    out = torch.zeros(*g.shape[:-2], h, w, dtype=g.dtype, device=g.device)
    out.index_add_(-2, y0, tmp * ly0[:, None])
    out.index_add_(-2, y1, tmp * ly1[:, None])
    return out


def recon_tail_input_grad_closed_form(dec: Tensor, x: Tensor, g_spatial: Tensor, g_freq: Tensor,
                                      norm: Optional[str] = "ortho") -> Tensor:
    """d(sum_n g_spatial[n]*spatial[n] + g_freq[n]*freq[n]) / d x of O.recon_tail:
    g_x = -(gs*sign(d)/(C*H*W) + fft_r2c_backward(gf*sign(dF)/(C*H*Wh))), d = rec - x -- the full-resolution g_rec of
    O.recon_tail_backward_closed_form, negated, before any resize."""
    N, C = dec.shape[:2]
    H, W = x.shape[-2:]
    Wh = W // 2 + 1
    d = O.bilinear_align_corners(dec, (H, W)) - x
    D = O.cat_rfft2(d, norm)
    gs = (g_spatial / (C * H * W)).view(N, 1, 1, 1)
    gf = (g_freq / (C * H * Wh)).view(N, 1, 1, 1)
    return -(gs * torch.sign(d) + O.rfft2_grad_closed_form(gf * torch.sign(D), (H, W), norm))


def attention_prep_input_grad_closed_form(pred: Tensor, x: Tensor, size: Sequence[int], g_spat_diff: Optional[Tensor],
                                          g_freq_diff: Optional[Tensor], norm: Optional[str] = "ortho") -> Tensor:
    """d(sum g_spat_diff*spat_diff + g_freq_diff*freq_diff) / d x of O.attention_prep (pred is detached):
    g_d = sign(d)*g_sd + fft_r2c_backward(sign(F)*g_fd) at `size`, F = cat rfft2(d), d = down(pred) - down(x);
    g_x = -(transposed align-corners resize)(g_d)."""
    d = O.bilinear_align_corners(pred, size) - O.bilinear_align_corners(x, size)
    g_d = torch.zeros_like(d)
    if g_spat_diff is not None:
        g_d = g_d + torch.sign(d) * g_spat_diff
    if g_freq_diff is not None:
        g_d = g_d + O.rfft2_grad_closed_form(torch.sign(O.cat_rfft2(d, norm)) * g_freq_diff, size, norm)
    return -bilinear_align_corners_transpose(g_d, x.shape[-2:])


def dynamic_filter_diff_grad_closed_form(x: Tensor, diff: Tensor, w1: Tensor, bn_gamma: Tensor, bn_beta: Tensor,
                                         w2: Tensor, act: str, g_mask: Optional[Tensor], g_filtered: Optional[Tensor],
                                         training: bool = True, running_mean: Optional[Tensor] = None,
                                         running_var: Optional[Tensor] = None) -> Tensor:
    """d(sum g_mask*mask + g_filtered*(mask*x)) / d diff of O.dynamic_filter: the guide channels enter only the 1x1
    layer2 conv, so g_diff[n,k,p] = w2[2+k] * g_logit[n,p], g_logit = (g_mask + sum_c g_filtered*x) * m(1-m)."""
    with torch.no_grad():
        mask, _, _ = O.dynamic_filter(x, diff, w1, bn_gamma, bn_beta, w2, act, training, running_mean, running_var)
    g = torch.zeros_like(mask)
    if g_mask is not None:
        g = g + g_mask
    if g_filtered is not None:
        g = g + (g_filtered * x).sum(dim=1, keepdim=True)
    g_logit = g * mask * (1 - mask)
    return w2.reshape(-1)[2:].view(1, -1, 1, 1) * g_logit
