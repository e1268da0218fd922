"""a1 parity: CUDA recon tail (through the C ABI) vs the oracle and vs reference fixtures."""
import math

import pytest
import torch

from oracle import recon_path as O

pytestmark = pytest.mark.gpu

SHAPES = [
    # N, C, h, w, H, W
    (2, 3, 10, 10, 20, 20),      # dynamic plan 5*4
    (2, 3, 5, 6, 11, 12),        # prime 11 rows / 3*4 cols, non-square
    (3, 2, 8, 12, 16, 24),
    (1, 3, 19, 19, 38, 38),      # 19*2
    (2, 3, 38, 38, 76, 76),
    (1, 1, 7, 9, 21, 15),        # odd sizes: no Nyquist column
    (2, 3, 128, 128, 256, 256),  # UDR18 / UDR50 config (static plan)
    (1, 3, 112, 112, 224, 224),
    (1, 3, 150, 150, 299, 299),  # 13*23
    (2, 3, 192, 192, 380, 380),  # UDEB4 config (static plan 19*5*4)
    (1, 3, 200, 100, 50, 40),    # downsampling path of the transposed resize
    (2, 3, 29, 29, 58, 58),      # 58 = 2*29: Bluestein (prime factor > 23) on both axes
    (1, 2, 31, 40, 62, 80),      # Bluestein columns (62 = 2*31), mixed-radix rows
    (1, 3, 124, 124, 248, 248),  # the ADVICE example: 248 = 8*31
    (1, 1, 20, 37, 40, 37),      # prime 37 rows
    (1, 3, 128, 150, 256, 300),  # first-generation kernels with 256-point columns (300 is no second-generation size)
    (1, 3, 150, 190, 300, 380),  # first-generation kernels with 380-point rows
]


def _inputs(shape, seed=0):
    N, C, h, w, H, W = shape
    g = torch.Generator().manual_seed(seed)
    dec = torch.tanh(torch.randn(N, C, h, w, generator=g))
    x = torch.rand(N, C, H, W, generator=g) * 2 - 1
    return dec, x


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("norm", ["ortho", None])
def test_forward_vs_oracle(shape, norm):
    from unidefense_b200 import ops
    dec, x = _inputs(shape)
    rec, sp, fr = ops.recon_tail(dec.cuda(), x.cuda(), norm)
    rec64, sp64, fr64 = O.recon_tail(dec.double(), x.double(), norm)
    # (the fp64 oracle also evaluates the resize coordinates in fp64; ATen and the kernel use fp32)
    torch.testing.assert_close(rec.cpu().double(), rec64, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(sp.cpu().double(), sp64, rtol=1e-4, atol=1e-7)
    torch.testing.assert_close(fr.cpu().double(), fr64, rtol=1e-4, atol=1e-7)
    # and against the fp32 two-FFT formulation the reference actually runs
    rec32, sp32, fr32 = O.recon_tail(dec, x, norm)
    torch.testing.assert_close(rec.cpu(), rec32, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(sp.cpu(), sp32, rtol=1e-4, atol=1e-7)
    torch.testing.assert_close(fr.cpu(), fr32, rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("shape", SHAPES)
def test_backward_vs_oracle(shape):
    from unidefense_b200 import ops
    N, C, h, w, H, W = shape
    dec, x = _inputs(shape, seed=1)
    g = torch.Generator().manual_seed(5)
    gs = torch.rand(N, generator=g) + 0.5
    gf = torch.rand(N, generator=g) + 0.5
    if N > 1:                      # the engine's fake rows: zero upstream grad
        gs[-1] = 0.0
        gf[-1] = 0.0
    d = dec.cuda().requires_grad_()
    _, sp, fr = ops.recon_tail(d, x.cuda(), "ortho")
    (sp * gs.cuda()).sum().add((fr * gf.cuda()).sum()).backward()
    got = d.grad.cpu().double()

    d64 = dec.double().requires_grad_()
    rec64, sp64, fr64 = O.recon_tail(d64, x.double(), "ortho")
    ((sp64 * gs.double()).sum() + (fr64 * gf.double()).sum()).backward()
    want = d64.grad
    # |.| is not differentiable at 0: bins whose magnitude is at fp32 noise level may legitimately
    # take either sign.  Give each such bin its worst-case contribution as extra budget.
    with torch.no_grad():
        dd = rec64 - x.double()
        D = O.cat_rfft2(dd, "ortho")
        Wh = W // 2 + 1
        up = math.ceil(H / h) * math.ceil(W / w) + 1
        for n in range(N):
            amb_f = int((D[n].abs() < 2e-5 * max(float(D[n].abs().max()), 1e-30)).sum())
            amb_s = int((dd[n].abs() < 2e-6).sum())
            budget = (amb_f * 2 * float(gf[n]) / (C * H * Wh) / math.sqrt(H * W) * up
                      + amb_s * 2 * float(gs[n]) / (C * H * W) * up)
            tol = 1e-4 * float(want[n].abs().max()) + budget + 1e-12
            err = float((got[n] - want[n]).abs().max())
            assert err <= tol, f"sample {n}: err {err:.3e} > tol {tol:.3e} (ambiguous bins f={amb_f} s={amb_s})"
    if N > 1:
        assert float(got[-1].abs().max()) == 0.0
    # closed-form oracle agrees too
    cf = O.recon_tail_backward_closed_form(dec.double(), x.double(), gs.double(), gf.double())
    torch.testing.assert_close(cf, want, rtol=1e-8, atol=1e-10)


def test_against_reference_fixture(golden_path):
    """rec / spatial / freq captured inside the reference model classes' forward()."""
    from unidefense_b200 import ops
    fix = golden_path
    nblocks = 2 if fix["arch"] == "r18" else 3
    dec = fix[f"dec_out{nblocks}"]
    rec, sp, fr = ops.recon_tail(dec.cuda(), fix["x"].cuda(), "ortho")
    torch.testing.assert_close(rec.cpu(), fix["rec"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(sp.cpu(), fix["spatial"], rtol=1e-4, atol=1e-7)
    torch.testing.assert_close(fr.cpu(), fix["freq"], rtol=1e-4, atol=1e-7)


def test_empty_and_errors():
    from unidefense_b200 import ops
    dec = torch.zeros(0, 3, 4, 4, device="cuda")
    x = torch.zeros(0, 3, 8, 8, device="cuda")
    rec, sp, fr = ops.recon_tail(dec, x)
    assert rec.shape == (0, 3, 8, 8) and sp.numel() == 0 and fr.numel() == 0
    with pytest.raises(RuntimeError):
        ops.recon_tail(torch.zeros(1, 1, 8, 8, device="cuda"), torch.zeros(1, 1, 8, 1025, device="cuda"))   # > UD_FFT_MAX_N
    with pytest.raises(RuntimeError):
        ops.recon_tail(torch.zeros(1, 3, 4, 4), torch.zeros(1, 3, 8, 8))  # CPU tensors: no fallback


def test_linearity_property_full_size():
    """Size-independent property at the BASELINE config shape (N=32, 380^2): the freq loss of
    (dec, x) with x := rec (zero difference) is exactly 0 and scaling the difference scales
    both losses linearly."""
    from unidefense_b200 import ops
    g = torch.Generator().manual_seed(3)
    dec = torch.tanh(torch.randn(32, 3, 192, 192, generator=g)).cuda()
    x = (torch.rand(32, 3, 380, 380, generator=g) * 2 - 1).cuda()
    rec, sp, fr = ops.recon_tail(dec, x)
    _, sp0, fr0 = ops.recon_tail(dec, rec)
    assert float(sp0.abs().max()) == 0.0 and float(fr0.abs().max()) == 0.0
    # x' = rec - 2*(rec - x)  => d' = 2 d
    _, sp2, fr2 = ops.recon_tail(dec, rec - 2.0 * (rec - x))
    torch.testing.assert_close(sp2, 2 * sp, rtol=1e-5, atol=0)
    torch.testing.assert_close(fr2, 2 * fr, rtol=1e-5, atol=0)
    # Parseval: sum |D|^2 == sum d^2 (ortho) bounds the L1 spectrum: freq*C*H*Wh <= sqrt(2*bins*energy)
    assert torch.isfinite(fr).all() and (fr > 0).all()


def test_rec_output_is_differentiable():
    """out['rec'] = interpolate(dec) carries a gradient in the reference (model/unidefense.py:244): a loss on it must
    reach dec (transposed bilinear resize), alone and together with the spatial/freq terms."""
    from unidefense_b200 import ops
    g = torch.Generator().manual_seed(11)
    dec = torch.tanh(torch.randn(2, 3, 19, 23, generator=g))
    x = torch.rand(2, 3, 38, 40, generator=g) * 2 - 1
    gr = torch.randn(2, 3, 38, 40, generator=g)
    for with_losses in (False, True):
        d = dec.cuda().requires_grad_()
        rec, sp, fr = ops.recon_tail(d, x.cuda())
        loss = (rec * gr.cuda()).sum() + ((0.3 * sp.sum() + fr.sum()) if with_losses else 0.0)
        loss.backward()
        d64 = dec.double().requires_grad_()
        rec64, sp64, fr64 = O.recon_tail(d64, x.double())
        loss64 = (rec64 * gr.double()).sum() + ((0.3 * sp64.sum() + fr64.sum()) if with_losses else 0.0)
        loss64.backward()
        torch.testing.assert_close(d.grad.cpu().double(), d64.grad, rtol=1e-4, atol=1e-5 * float(d64.grad.abs().max()))


def test_unsupported_norm_is_rejected():
    from unidefense_b200 import ops
    with pytest.raises(ValueError, match="freq_norm"):
        ops.recon_tail(torch.zeros(1, 3, 4, 4, device="cuda"), torch.zeros(1, 3, 8, 8, device="cuda"), norm="forward")
