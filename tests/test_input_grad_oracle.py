"""CPU: the closed forms of oracle/input_grad.py equal torch autograd of the oracle's forwards in fp64 (the forwards
are pinned to the live reference's fixtures, so their autograd stands for the reference's x gradient)."""
import pytest
import torch

from oracle import input_grad as G
from oracle import recon_path as O


def _gen(seed):
    return torch.Generator().manual_seed(seed)


@pytest.mark.parametrize("shape", [(2, 3, 10, 10, 20, 20), (1, 2, 5, 6, 11, 12), (2, 3, 20, 15, 10, 8),
                                   (1, 3, 19, 19, 38, 38)])
@pytest.mark.parametrize("norm", ["ortho", None])
def test_recon_tail_input_grad(shape, norm):
    N, C, h, w, H, W = shape
    g = _gen(1)
    dec = torch.tanh(torch.randn(N, C, h, w, generator=g, dtype=torch.float64))
    x = (torch.rand(N, C, H, W, generator=g, dtype=torch.float64) * 2 - 1).requires_grad_()
    gs = torch.rand(N, generator=g, dtype=torch.float64) + 0.5
    gf = torch.rand(N, generator=g, dtype=torch.float64) + 0.5
    if N > 1:
        gs[-1] = gf[-1] = 0.0
    _, sp, fr = O.recon_tail(dec, x, norm)
    ((sp * gs).sum() + (fr * gf).sum()).backward()
    cf = G.recon_tail_input_grad_closed_form(dec, x.detach(), gs, gf, norm)
    torch.testing.assert_close(cf, x.grad, rtol=1e-9, atol=1e-12)
    if N > 1:
        assert float(cf[-1].abs().max()) == 0.0


@pytest.mark.parametrize("R,h", [((38, 38), (12, 12)), ((32, 32), (8, 8)), ((20, 28), (6, 9)), ((8, 8), (4, 4)),
                                 ((5, 7), (9, 12))])
@pytest.mark.parametrize("which", ["sd", "fd", "both"])
def test_attention_prep_input_grad(R, h, which):
    g = _gen(2)
    N, C = 2, 3
    pred = torch.tanh(torch.randn(N, C, 16, 14, generator=g, dtype=torch.float64))
    x = (torch.rand(N, C, *R, generator=g, dtype=torch.float64) * 2 - 1).requires_grad_()
    gsd = torch.randn(N, C, *h, generator=g, dtype=torch.float64) if which != "fd" else None
    gfd = torch.randn(N, 2 * C, h[0], h[1] // 2 + 1, generator=g, dtype=torch.float64) if which != "sd" else None
    for norm in ("ortho", None):
        x.grad = None
        sd, fd = O.attention_prep(pred, x, h, norm)
        loss = (sd * gsd).sum() if gsd is not None else 0.0
        loss = loss + ((fd * gfd).sum() if gfd is not None else 0.0)
        loss.backward()
        cf = G.attention_prep_input_grad_closed_form(pred, x.detach(), h, gsd, gfd, norm)
        torch.testing.assert_close(cf, x.grad, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("kind", ["freq", "spat"])
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("bias", [False, True])
def test_dynamic_filter_diff_grad(kind, training, bias):
    g = _gen(3)
    N, C, hh, ww = 3, 8, 6, 5
    D = 6 if kind == "freq" else 3
    k = 1 if kind == "freq" else 3
    dt = torch.float64
    x = torch.randn(N, C, hh, ww, generator=g, dtype=dt)
    diff = torch.rand(N, D, hh, ww, generator=g, dtype=dt)
    if bias:                                    # model/modules.py: the bias rides on a constant-one guide channel
        diff = torch.cat([diff, torch.ones_like(diff[:, :1])], dim=1)
    diff.requires_grad_()
    w1 = torch.randn(C, C, k, k, generator=g, dtype=dt) * 0.3
    gamma, beta = torch.rand(C, generator=g, dtype=dt) + 0.5, torch.randn(C, generator=g, dtype=dt) * 0.1
    w2 = torch.randn(1, 2 + diff.shape[1], 1, 1, generator=g, dtype=dt)
    rm, rv = torch.randn(C, generator=g, dtype=dt) * 0.1, torch.rand(C, generator=g, dtype=dt) + 0.5
    gm = torch.randn(N, 1, hh, ww, generator=g, dtype=dt)
    gfilt = torch.randn(N, C, hh, ww, generator=g, dtype=dt)
    mask, filt, _ = O.dynamic_filter(x, diff, w1, gamma, beta, w2, "swish", training, rm, rv)
    ((mask * gm).sum() + (filt * gfilt).sum()).backward()
    cf = G.dynamic_filter_diff_grad_closed_form(x, diff.detach(), w1, gamma, beta, w2, "swish", gm, gfilt, training,
                                                rm, rv)
    torch.testing.assert_close(cf, diff.grad, rtol=1e-9, atol=1e-12)


def test_bilinear_transpose_is_the_adjoint():
    g = _gen(4)
    for (h, w), (H, W) in (((7, 9), (3, 4)), ((3, 4), (7, 9)), ((1, 5), (4, 1))):
        a = torch.randn(2, h, w, generator=g, dtype=torch.float64)
        b = torch.randn(2, H, W, generator=g, dtype=torch.float64)
        lhs = (O.bilinear_align_corners(a, (H, W)) * b).sum()
        rhs = (a * G.bilinear_align_corners_transpose(b, (h, w))).sum()
        torch.testing.assert_close(lhs, rhs, rtol=1e-12, atol=1e-12)
