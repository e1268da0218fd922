"""Every FFT length 1..1024 through every FFT entry point, against torch.fft in fp64.

The 2-D real FFT runs on five line-FFT engines: the small-plane DFT (ud_attention.cu), the two-kernel Stockham path
(ud_fft2d.cu), the recon tail's first and second generation and the frequency style transfer.  Each runs mixed radix
for lengths whose prime factors are <= 23 and Bluestein at a power-of-two working length m >= 2n - 1 otherwise.  A
wrong twiddle index in one radix stage, an off-by-one in one column tile or in the Bluestein wrap shows at a few lengths
only, so each test walks one band of lengths through one engine, gathers every failing length with its error and asserts
once, so that one run shows the whole failing set.  The per-shape tests of the other modules stay as they are.

Tolerance: the suite's close (rtol 1e-4, atol 1e-5 max|ref|) on every output, plus a normwise relative error
||got - ref||_2 / ||ref||_2 <= 1e-5 on every FFT output.  The indexing slips this file targets give O(1) errors.
"""
import math
import zlib

import pytest
import torch

from oracle import recon_path as O

BANDS = [(1, 64), (65, 256), (257, 512), (513, 1024)]
BAND_IDS = [f"{a}-{b}" for a, b in BANDS]
# the static plans' lengths, the steps of the Bluestein working length (m = 512 from 257, m = 1024 from 513), the
# largest prime (m = 2048) and the largest length
BOUNDARY = (224, 256, 257, 299, 380, 512, 513, 1021, 1024)
NORMWISE = 1e-5
NC = (2, 2)                      # samples, channels: several planes per launch, still cheap at every length


def _band(band):
    return range(band[0], band[1] + 1)


class _Sweep:
    """Collects the failing cases of one (engine, band) and the largest normwise error met."""

    def __init__(self, name):
        self.name = name
        self.failures = []
        self.worst = 0.0

    def check(self, what, got, ref, rtol=1e-4, atol=None, normwise=True):
        got = got.detach().cpu().to(ref.dtype)
        ref = ref.detach()
        ref_max = float(ref.abs().max()) if ref.numel() else 0.0
        atol = 1e-5 * max(ref_max, 1e-6) if atol is None else atol
        err = (got - ref).abs()
        bad = int((~(err <= atol + rtol * ref.abs())).sum())           # NaN counts as bad
        rnorm = float(ref.norm())
        rel = float((got - ref).norm()) / rnorm if rnorm > 0 else float((got - ref).norm())
        if normwise and rel == rel:
            self.worst = max(self.worst, rel)
        if bad:
            self.failures.append(f"{what}: {bad}/{ref.numel()} elements off, max err {float(err.max()):.3e} "
                                 f"(max|ref| {ref_max:.3e}), normwise {rel:.3e}")
        elif normwise and not rel <= NORMWISE:
            self.failures.append(f"{what}: normwise error {rel:.3e} > {NORMWISE:.0e}")

    def run(self, what, fn, *args):
        try:
            fn(self, what, *args)
        except RuntimeError as e:                # an entry point rejected the size
            self.failures.append(f"{what}: {str(e).splitlines()[0]}")

    def finish(self):
        print(f"\n{self.name}: max normwise error {self.worst:.3e}, {len(self.failures)} failing")
        assert not self.failures, (f"{self.name}: {len(self.failures)} failing case(s):\n  "
                                   + "\n  ".join(self.failures))


def _gen(*key):
    return torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))


# ---------------------------------------------------------------------------------------------- ud_rfft2 / ud_irfft2
def _rfft2_pair(sw, what, shape, norm):
    """forward and inverse plus both adjoints through backward, as test_rfft2_irfft2_fwd_bwd does"""
    from unidefense_b200 import ops
    N, C, h, w = shape
    g = _gen("rfft2", shape, norm)
    x = torch.randn(N, C, h, w, generator=g)
    wgt = torch.randn(N, 2 * C, h, w // 2 + 1, generator=g)
    xc = x.cuda().requires_grad_()
    xf = ops.rfft2_cat(xc, norm)
    (xf * wgt.cuda()).sum().backward()
    x64 = x.double().requires_grad_()
    xf64 = O.cat_rfft2(x64, norm)
    (xf64 * wgt.double()).sum().backward()
    sw.check(f"{what} rfft2", xf, xf64)
    sw.check(f"{what} rfft2 adjoint", xc.grad, x64.grad)

    z = torch.randn(N, 2 * C, h, w // 2 + 1, generator=g)
    gy = torch.randn(N, C, h, w, generator=g)
    zc = z.cuda().requires_grad_()
    y = ops.irfft2_cat(zc, (h, w), norm)
    (y * gy.cuda()).sum().backward()
    z64 = z.double().requires_grad_()
    y64 = O.irfft2_from_cat(z64, (h, w), norm)
    (y64 * gy.double()).sum().backward()
    sw.check(f"{what} irfft2", y, y64)
    sw.check(f"{what} irfft2 adjoint", zc.grad, z64.grad)


def _rfft2_sweep(name, band, shape_of):
    sw = _Sweep(name)
    for n in _band(band):
        shape = shape_of(n)
        sw.run(f"n={n} {shape} ortho", _rfft2_pair, shape, "ortho")
        if n in BOUNDARY:
            sw.run(f"n={n} {shape} norm=None", _rfft2_pair, shape, None)
    sw.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("band", BANDS, ids=BAND_IDS)
def test_rfft2_two_kernel_columns(band):
    """column length n; the 65-point rows force the two-kernel path at every n"""
    _rfft2_sweep(f"rfft2 two-kernel columns {band}", band, lambda n: (*NC, n, 65))


@pytest.mark.gpu
@pytest.mark.parametrize("band", BANDS, ids=BAND_IDS)
def test_rfft2_two_kernel_rows(band):
    _rfft2_sweep(f"rfft2 two-kernel rows {band}", band, lambda n: (*NC, 65, n))


SMALL_PARTNERS = (1, 2, 31, 61, 64)


@pytest.mark.gpu
def test_rfft2_small_plane():
    """planes with h, w <= 64 run the one-CTA-per-plane DFT of ud_attention.cu: every length against a few partners"""
    sw = _Sweep("rfft2 small-plane 1-64")
    for n in range(1, 65):
        for p in SMALL_PARTNERS:
            sw.run(f"{n}x{p}", _rfft2_pair, (*NC, n, p), "ortho")
            sw.run(f"{p}x{n}", _rfft2_pair, (*NC, p, n), "ortho")
    sw.finish()


def _attn_prep_case(sw, what, h, w):
    """x at (2h-1, 2w-1) and pred at (h, w) make every align_corners coordinate exact in fp32, so the kernel and the
    fp64 oracle sample the same pixels and only the transform's rounding is left"""
    from unidefense_b200 import ops
    N, C = NC
    g = _gen("attn_prep", h, w)
    pred = torch.tanh(torch.randn(N, C, h, w, generator=g))
    x = torch.rand(N, C, 2 * h - 1, 2 * w - 1, generator=g) * 2 - 1
    gfd = torch.randn(N, 2 * C, h, w // 2 + 1, generator=g)
    for norm in ("ortho", None):
        xc = x.cuda().requires_grad_()
        sd, fd = ops.attn_prep(pred.cuda(), xc, (h, w), norm)
        (fd * gfd.cuda()).sum().backward()
        x64 = x.double().requires_grad_()
        sd64, fd64 = O.attention_prep(pred.double(), x64, (h, w), norm)
        (fd64 * gfd.double()).sum().backward()
        sw.check(f"{what} {norm} spat_diff", sd, sd64, normwise=False)
        sw.check(f"{what} {norm} freq_diff", fd, fd64)
        # |.| has a kink at 0: a bin at fp32 noise level may take either sign; budget its full contribution
        with torch.no_grad():
            Fd = O.cat_rfft2(O.bilinear_align_corners(pred.double(), (h, w)) - O.bilinear_align_corners(x.double(), (h, w)),
                             norm)
            amb_f = int((Fd.abs() < 2e-5 * float(Fd.abs().max())).sum())
            nrm = 1.0 / math.sqrt(h * w) if norm == "ortho" else 1.0
            budget = amb_f * 2 * nrm * float(gfd.abs().max())
        err = float((xc.grad.cpu().double() - x64.grad).abs().max())
        tol = 1e-4 * float(x64.grad.abs().max()) + budget + 1e-9
        if not err <= tol:
            sw.failures.append(f"{what} {norm} x-gradient: err {err:.3e} > tol {tol:.3e} (ambiguous bins {amb_f})")


@pytest.mark.gpu
def test_attn_prep_prime_planes():
    """ud_attn_prep(_bwd) share at_r2c_plane with the small-plane rfft2: primes 29..61 the size sets above miss"""
    sw = _Sweep("attn_prep small-plane primes")
    for h, w in ((29, 29), (31, 37), (61, 61)):
        sw.run(f"{h}x{w}", _attn_prep_case, h, w)
    sw.finish()


def _mask_case(sw, what, shape, norm):
    from unidefense_b200 import ops
    N, C, H, W = shape
    g = _gen("mask", shape, norm)
    x = torch.randn(shape, generator=g)
    mask = torch.rand(N, H, W // 2 + 1, generator=g)
    y = ops.spectral_mask_filter(x.cuda(), mask.cuda(), norm)
    sw.check(what, y, O.spectral_mask_filter(x.double(), mask.double(), norm))


@pytest.mark.gpu
def test_spectral_mask_filter_boundary_lengths():
    """mask folded into the inverse's load, at the static lengths and the Bluestein working-length steps"""
    sw = _Sweep("spectral_mask_filter boundary lengths")
    for n in BOUNDARY:
        for shape in ((*NC, n, 65), (*NC, 65, n)):
            for norm in ("ortho", None):
                sw.run(f"n={n} {shape} {norm}", _mask_case, shape, norm)
    sw.finish()


# ---------------------------------------------------------------------------------------------- recon tail
def _sign_budget(dd, D, rec_err, gs, gf, C, H, W, up):
    """|.| is not differentiable at 0: a pixel or bin whose value lies within the kernel's rounding of 0 may take either
    sign.  Give each such one its worst-case contribution, per sample.  `rec_err` widens the bands by what the kernel's
    fp32 resize coordinates move rec (the oracle computes them in fp64)."""
    Wh = W // 2 + 1
    out = []
    for n in range(dd.shape[0]):
        thr_f = 2e-5 * max(float(D[n].abs().max()), 1e-30) + float(rec_err[n].abs().sum()) / math.sqrt(H * W)
        amb_f = int((D[n].abs() < thr_f).sum())
        amb_s = int((dd[n].abs() < 2e-6 + rec_err[n]).sum())
        out.append((amb_f * 2 * float(gf[n]) / (C * H * Wh) / math.sqrt(H * W) + amb_s * 2 * float(gs[n]) / (C * H * W))
                   * up)
    return out


def _recon_case(sw, what, h, w, H, W, grad_x=True):
    """forward (rec, spatial, freq) and the backward to dec and (grad_x) to x, ortho, against the fp64 oracle.
    Without grad_x the backward runs the training-path kernels (g_x == NULL)."""
    from unidefense_b200 import ops
    N, C = NC
    g = _gen("recon", h, w, H, W)
    dec = torch.tanh(torch.randn(N, C, h, w, generator=g))
    x = torch.rand(N, C, H, W, generator=g) * 2 - 1
    gs = torch.rand(N, generator=g) + 0.5
    gf = torch.rand(N, generator=g) + 0.5
    d = dec.cuda().requires_grad_()
    xc = x.cuda().requires_grad_(grad_x)
    rec, sp, fr = ops.recon_tail(d, xc, "ortho")
    (sp * gs.cuda()).sum().add((fr * gf.cuda()).sum()).backward()
    d64 = dec.double().requires_grad_()
    x64 = x.double().requires_grad_(grad_x)
    rec64, sp64, fr64 = O.recon_tail(d64, x64, "ortho")
    ((sp64 * gs.double()).sum() + (fr64 * gf.double()).sum()).backward()
    # tolerances of test_forward_vs_oracle; rec is a resize, not a transform: no normwise bound
    sw.check(f"{what} rec", rec, rec64, atol=1e-4, normwise=False)
    sw.check(f"{what} spatial", sp, sp64, atol=1e-7)
    sw.check(f"{what} freq", fr, fr64, atol=1e-7)
    with torch.no_grad():
        dd = rec64 - x64
        D = O.cat_rfft2(dd, "ortho")
        rec_err = (rec.detach().cpu().double() - rec64).abs()
        up = math.ceil(H / h) * math.ceil(W / w) + 1
        grads = [("g_dec", d.grad, d64.grad, up)] + ([("g_x", xc.grad, x64.grad, 1)] if grad_x else [])
        if not grad_x and xc.grad is not None:
            sw.failures.append(f"{what}: x got a gradient it did not ask for")
        for name, got, want, u in grads:
            budget = _sign_budget(dd, D, rec_err, gs, gf, C, H, W, u)
            got = got.cpu().double()
            for n in range(N):
                tol = 1e-4 * float(want[n].abs().max()) + budget[n] + 1e-12
                err = float((got[n] - want[n]).abs().max())
                if not err <= tol:
                    sw.failures.append(f"{what} {name} sample {n}: err {err:.3e} > tol {tol:.3e}")


def _half(n):
    return (n + 1) // 2


@pytest.mark.gpu
@pytest.mark.parametrize("band", BANDS, ids=BAND_IDS)
def test_recon_tail_columns(band):
    """column length H at W = 20: every H runs the first-generation kernels (the second needs both sides configured)"""
    sw = _Sweep(f"recon_tail columns {band}")
    for n in _band(band):
        sw.run(f"H={n} W=20", _recon_case, _half(n), 10, n, 20)
    sw.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("band", BANDS, ids=BAND_IDS)
def test_recon_tail_rows(band):
    sw = _Sweep(f"recon_tail rows {band}")
    for n in _band(band):
        sw.run(f"H=20 W={n}", _recon_case, 10, _half(n), 20, n)
    sw.finish()


@pytest.mark.gpu
def test_recon_tail_large_planes():
    """Square planes of Bluestein (372 = 4*3*31) and mixed-radix (1024) length; full-width decoders (w = W) at the
    longest rows; a row length whose full-width decoder leaves less free shared memory at 12 row pairs than the kernels'
    static bytes (402); a decoder twice as wide as the tightest rows (2045 -> 1023, an exact resize).  The largest
    Bluestein shapes also run the training-path backward (no x gradient)."""
    sw = _Sweep("recon_tail large planes")
    for h, w, H, W in ((186, 186, 372, 372), (512, 512, 1024, 1024), (10, 1021, 20, 1021), (10, 1024, 20, 1024),
                       (10, 402, 20, 402), (10, 2045, 20, 1023)):
        sw.run(f"dec {h}x{w} -> {H}x{W}", _recon_case, h, w, H, W)
    for h, w, H, W in ((186, 186, 372, 372), (10, 511, 20, 1021), (10, 1021, 20, 1021)):
        sw.run(f"dec {h}x{w} -> {H}x{W} no x gradient", _recon_case, h, w, H, W, False)
    sw.finish()


# ---------------------------------------------------------------------------------------------- frequency style
def _freq_style_case(sw, what, H, W):
    from unidefense_b200 import ops
    N, C = NC
    g = _gen("freq_style", H, W)
    content = torch.rand(N, C, H, W, generator=g) * 2 - 1
    style = torch.rand(N, C, H, W, generator=g) * 2 - 1
    lm = torch.rand(N, generator=g) / 2 + 0.5
    y = ops.freq_style_transfer(content.cuda(), style.cuda(), lm.cuda())
    y64 = O.frequency_style_transfer(content.double(), style.double(), lm.double().view(-1, 1, 1, 1))
    sw.check(what, y, y64)


@pytest.mark.gpu
@pytest.mark.parametrize("band", BANDS, ids=BAND_IDS)
def test_freq_style_columns(band):
    sw = _Sweep(f"freq_style columns {band}")
    for n in _band(band):
        sw.run(f"H={n} W=20", _freq_style_case, n, 20)
    sw.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("band", BANDS, ids=BAND_IDS)
def test_freq_style_rows(band):
    sw = _Sweep(f"freq_style rows {band}")
    for n in _band(band):
        sw.run(f"H=20 W={n}", _freq_style_case, 20, n)
    sw.finish()


@pytest.mark.gpu
def test_freq_style_large_planes():
    sw = _Sweep("freq_style large planes")
    for n in (372, 1024):
        sw.run(f"{n}x{n}", _freq_style_case, n, n)
    sw.finish()


# ---------------------------------------------------------------------------------------------- size predicates
def _smooth(n):
    for p in (2, 3, 5, 7, 11, 13, 17, 19, 23):
        while n % p == 0:
            n //= p
    return n == 1


def test_fft_size_predicates():
    """mixed radix exactly for 1 <= n <= 1024 with every prime factor <= 23; some plan for every 1 <= n <= 1024"""
    from unidefense_b200 import _lib
    L = _lib.lib()
    wrong = []
    for n in range(0, 1101):
        if L.ud_fft_size_supported(n) != int(1 <= n <= 1024 and _smooth(n)):
            wrong.append(f"ud_fft_size_supported({n}) = {L.ud_fft_size_supported(n)}")
        if L.ud_fft_size_any(n) != int(1 <= n <= 1024):
            wrong.append(f"ud_fft_size_any({n}) = {L.ud_fft_size_any(n)}")
    assert not wrong, "\n".join(wrong)
