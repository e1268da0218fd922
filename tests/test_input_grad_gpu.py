"""Gradients with respect to the input image x: every route by which x reaches the outputs in the reference (backbone,
attention error maps -> dynamic-filter guide channels, reconstruction losses, pass-2 blur / downscale) against torch
autograd of the oracle's op sequence."""
import math
import os

import pytest
import torch
import torch.nn.functional as F

import procedural as P
from oracle import input_grad as G
from oracle import recon_path as O
from oracle import ref_model
from test_recon_tail_gpu import SHAPES, _inputs

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _rel2(a, b):
    return float((a.detach().cpu().double() - b.detach().cpu().double()).norm() / b.detach().cpu().double().norm())


# ---------------------------------------------------------------------------------------------- reconstruction tail
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("norm", ["ortho", None])
def test_recon_tail_x_grad(shape, norm):
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
    xc = x.cuda().requires_grad_()
    _, sp, fr = ops.recon_tail(d, xc, norm)
    (sp * gs.cuda()).sum().add((fr * gf.cuda()).sum()).backward()
    got = xc.grad.cpu().double()

    d64 = dec.double().requires_grad_()
    x64 = x.double().requires_grad_()
    rec64, sp64, fr64 = O.recon_tail(d64, x64, norm)
    ((sp64 * gs.double()).sum() + (fr64 * gf.double()).sum()).backward()
    want = x64.grad
    torch.testing.assert_close(G.recon_tail_input_grad_closed_form(dec.double(), x.double(), gs.double(), gf.double(),
                                                                   norm), want, rtol=1e-8, atol=1e-12)
    # the |.|-kink budget of test_backward_vs_oracle, without the resize fan-in: g_x is the full-resolution g_rec
    nrm = 1.0 / math.sqrt(H * W) if norm == "ortho" else 1.0
    with torch.no_grad():
        dd = rec64 - x64
        D = O.cat_rfft2(dd, norm)
        Wh = W // 2 + 1
        for n in range(N):
            amb_f = int((D[n].abs() < 2e-5 * max(float(D[n].abs().max()), 1e-30)).sum())
            amb_s = int((dd[n].abs() < 2e-6).sum())
            budget = amb_f * 2 * float(gf[n]) / (C * H * Wh) * nrm + amb_s * 2 * float(gs[n]) / (C * H * W)
            tol = 1e-4 * float(want[n].abs().max()) + budget + 1e-12
            err = float((got[n] - want[n]).abs().max())
            assert err <= tol, f"sample {n}: err {err:.3e} > tol {tol:.3e} (ambiguous bins f={amb_f} s={amb_s})"
    if N > 1:
        assert float(got[-1].abs().max()) == 0.0
    # the dec gradient of the g_x kernels equals the training path's
    d2 = dec.cuda().requires_grad_()
    _, sp2, fr2 = ops.recon_tail(d2, x.cuda(), norm)
    (sp2 * gs.cuda()).sum().add((fr2 * gf.cuda()).sum()).backward()
    torch.testing.assert_close(d.grad, d2.grad, rtol=1e-5, atol=1e-6 * float(d2.grad.abs().max()) + 1e-12)


@pytest.mark.parametrize("shape", [(2, 3, 192, 192, 380, 380), (2, 3, 29, 29, 58, 58), (1, 2, 31, 40, 62, 80)])
def test_recon_tail_x_grad_only_and_none(shape):
    """dec detached -> g_x alone (no transposed resize); x without grad -> None, and the training kernels."""
    from unidefense_b200 import ops
    dec, x = _inputs(shape, seed=2)
    dc, xc = dec.cuda(), x.cuda().requires_grad_()
    _, sp, fr = ops.recon_tail(dc, xc)
    (0.1 * sp.sum() + fr.sum()).backward()
    d_both = dc.clone().requires_grad_()
    x_both = x.cuda().requires_grad_()
    _, sp2, fr2 = ops.recon_tail(d_both, x_both)
    (0.1 * sp2.sum() + fr2.sum()).backward()
    assert torch.equal(xc.grad, x_both.grad)           # same kernel, same fixed-order arithmetic
    d3 = dc.clone().requires_grad_()
    x3 = x.cuda()
    _, sp3, fr3 = ops.recon_tail(d3, x3)
    (0.1 * sp3.sum() + fr3.sum()).backward()
    assert x3.grad is None and d3.grad is not None
    _, sp4, _ = ops.recon_tail(dc, x.cuda())
    assert sp4.grad_fn is None                          # nothing requires grad: no graph, no sign bytes


# ---------------------------------------------------------------------------------------------- error maps
PREP = [((380, 380), (12, 12)), ((256, 256), (8, 8)), ((256, 256), (16, 16)), ((380, 380), (24, 24)),
        ((64, 64), (4, 4)), ((300, 220), (10, 7)), ((24, 20), (40, 33))]      # last: upsampling, also accepted


@pytest.mark.parametrize("R,h", PREP)
@pytest.mark.parametrize("which", ["sd", "fd", "both"])
def test_attn_prep_x_grad(R, h, which):
    from unidefense_b200 import ops
    g = torch.Generator().manual_seed(R[0] + 7 * h[0] + len(which))
    N, C = 2, 3
    pred = torch.tanh(torch.randn(N, C, max(R[0] // 2, 2), max(R[1] // 2, 2), generator=g))
    x = torch.rand(N, C, *R, generator=g) * 2 - 1
    gsd = torch.randn(N, C, *h, generator=g) if which != "fd" else None
    gfd = torch.randn(N, 2 * C, h[0], h[1] // 2 + 1, generator=g) if which != "sd" else None
    for norm in ("ortho", None):
        grads = []
        for _ in range(2):
            xc = x.cuda().requires_grad_()
            sd, fd = ops.attn_prep(pred.cuda(), xc, h, norm)
            loss = (sd * gsd.cuda()).sum() if gsd is not None else 0.0
            loss = loss + ((fd * gfd.cuda()).sum() if gfd is not None else 0.0)
            loss.backward()
            grads.append(xc.grad)
        assert torch.equal(grads[0], grads[1]), "error-map backward is not bitwise reproducible"
        x64 = x.double().requires_grad_()
        sd64, fd64 = O.attention_prep(pred.double(), x64, h, norm)
        loss64 = (sd64 * gsd.double()).sum() if gsd is not None else 0.0
        loss64 = loss64 + ((fd64 * gfd.double()).sum() if gfd is not None else 0.0)
        loss64.backward()
        want = x64.grad
        torch.testing.assert_close(G.attention_prep_input_grad_closed_form(
            pred.double(), x.double(), h, None if gsd is None else gsd.double(), None if gfd is None else gfd.double(),
            norm), want, rtol=1e-8, atol=1e-12)
        # |.| kinks: a small pixel / bin at fp32 noise level may take the other sign; budget its full contribution
        with torch.no_grad():
            d = O.bilinear_align_corners(pred.double(), h) - O.bilinear_align_corners(x.double(), h)
            Fd = O.cat_rfft2(d, norm)
            nrm = 1.0 / math.sqrt(h[0] * h[1]) if norm == "ortho" else 1.0
            amb_s = int((d.abs() < 2e-6).sum()) if gsd is not None else 0
            amb_f = int((Fd.abs() < 2e-5 * float(Fd.abs().max())).sum()) if gfd is not None else 0
            budget = (amb_s * 2 * (float(gsd.abs().max()) if gsd is not None else 0.0)
                      + amb_f * 2 * nrm * (float(gfd.abs().max()) if gfd is not None else 0.0))
        err = float((grads[0].cpu().double() - want).abs().max())
        tol = 1e-4 * float(want.abs().max()) + budget + 1e-9
        assert err <= tol, f"norm={norm}: err {err:.3e} > tol {tol:.3e} (ambiguous s={amb_s} f={amb_f})"


def test_attn_prep_no_grad_paths():
    from unidefense_b200 import ops
    pred = torch.rand(2, 3, 16, 16, device="cuda")
    x = torch.rand(2, 3, 32, 32, device="cuda")
    sd, fd = ops.attn_prep(pred, x, (8, 8))
    assert sd.grad_fn is None and fd.grad_fn is None
    xr = x.clone().requires_grad_()
    sd2, fd2 = ops.attn_prep(pred.requires_grad_(), xr, (8, 8))
    assert torch.equal(sd, sd2.detach()) and torch.equal(fd, fd2.detach())
    fd2.sum().backward()
    assert pred.grad is None and xr.grad is not None            # pred is data, as in the reference


# ---------------------------------------------------------------------------------------------- dynamic filters
@pytest.mark.parametrize("kind", ["freq", "spat"])
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("bias", [False, True])
def test_dyfi_diff_grad(kind, training, bias):
    from unidefense_b200 import ops
    g = torch.Generator().manual_seed(31 + 2 * int(training) + int(bias) + (5 if kind == "spat" else 0))
    N, C, h, w = (4, 64, 12, 7) if kind == "freq" else (4, 48, 12, 12)
    D, k = (6, 1) if kind == "freq" else (3, 3)
    x = torch.randn(N, C, h, w, generator=g)
    diff = torch.rand(N, D, h, w, generator=g)
    if bias:                   # model/modules.py: a constant-one guide channel carries layer2's bias
        diff = torch.cat([diff, torch.ones_like(diff[:, :1])], dim=1)
    w1 = torch.randn(C, C, k, k, generator=g) / (C * k * k) ** 0.5
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1
    w2 = torch.randn(1, 2 + diff.shape[1], 1, 1, generator=g) * 0.5
    rmean, rvar = torch.randn(C, generator=g) * 0.2, torch.rand(C, generator=g) + 0.5
    gm = torch.randn(N, 1, h, w, generator=g)
    go = torch.randn(N, C, h, w, generator=g)

    xc, dc = x.cuda(), diff.cuda().requires_grad_()
    proj = F.conv2d(xc, w1.cuda(), None, 1, k // 2)
    if training:
        mean, m2 = ops.bn_local_stats(proj)
        var, count = m2 / (N * h * w), N * h * w
    else:
        mean, var, count = rmean.cuda(), rvar.cuda(), 0
    mask, out = ops.dyfi_mask(proj, mean, torch.rsqrt(var + 1e-5), gamma.cuda(), beta.cuda(), dc, w2.cuda(), xc, "swish",
                              count, True)
    ((mask * gm.cuda()).sum() + (out * go.cuda()).sum()).backward()

    d64 = diff.double().requires_grad_()
    m64, o64, _ = O.dynamic_filter(x.double(), d64, w1.double(), gamma.double(), beta.double(), w2.double(), "swish",
                                   training, rmean.double(), rvar.double())
    ((m64 * gm.double()).sum() + (o64 * go.double()).sum()).backward()
    want = d64.grad
    torch.testing.assert_close(G.dynamic_filter_diff_grad_closed_form(
        x.double(), diff.double(), w1.double(), gamma.double(), beta.double(), w2.double(), "swish", gm.double(),
        go.double(), training, rmean.double(), rvar.double()), want, rtol=1e-8, atol=1e-12)
    torch.testing.assert_close(dc.grad.cpu().double(), want, rtol=1e-3, atol=1e-4 * float(want.abs().max()))


# ---------------------------------------------------------------------------------------------- perturbations
@pytest.mark.parametrize("R", [380, 256, 95, 64])
def test_blur_and_downscale_x_grad(R):
    from unidefense_b200 import ops
    g = torch.Generator().manual_seed(R)
    x = torch.rand(2, 3, R, R - 3, generator=g) * 2 - 1
    gy = torch.randn(2, 3, R, R - 3, generator=g)
    for fn, ref in ((ops.gaussian_blur5, O.random_blur), (ops.downscale_nearest, O.downscale)):
        xc = x.cuda().requires_grad_()
        (fn(xc) * gy.cuda()).sum().backward()
        x64 = x.double().requires_grad_()
        (ref(x64) * gy.double()).sum().backward()
        torch.testing.assert_close(xc.grad.cpu().double(), x64.grad, rtol=1e-5, atol=1e-6)
        xc2 = x.cuda().requires_grad_()
        (fn(xc2) * gy.cuda()).sum().backward()
        assert torch.equal(xc.grad, xc2.grad)


# ---------------------------------------------------------------------------------------------- whole model
CTOR = {"eb4": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2, drop_rate=0.0, drop_connect_rate=0.0)),
        "r18": ("UDR18", dict(num_classes=2, drop_rate=0.0)),
        "r50": ("UDR50", dict(extractor="resnet50", num_classes=2, drop_rate=0.0))}


@pytest.fixture()
def no_dropout(monkeypatch):
    monkeypatch.setattr(F, "dropout", lambda t, p=0.5, training=True, inplace=False: t * 1.0)


def _models(arch):
    from unidefense_b200.model import load_model
    name, kw = CTOR[arch]
    model = load_model(name)(**kw)
    P.fill_state_dict_(model, salt=5)          # sf_coef / fuse_coef are not degenerate
    cpu = ref_model.build(arch, **kw)
    cpu.load_state_dict(model.state_dict())
    return model.cuda(), cpu


def _objective(out, labels, train, cross_entropy, triplet):
    if not train:                               # the detector's score (engines' validate()/test())
        return torch.softmax(out["cls_out"], dim=1)[:, 0].sum()
    ld = out["loss_dict"]
    nr = int((labels == 0).sum())
    tri = sum(triplet(f, labels) for f in ld["triplet"])
    return (cross_entropy(out["cls_out"], labels) + 0.1 * ld["freq_mask"].mean() + 0.1 * ld["spat_mask"].mean()
            + 0.1 * tri + 0.1 * ld["spatial"][:nr].mean() + 1.0 * ld["freq"][:nr].mean())


@pytest.mark.parametrize("arch", ["eb4", "r18", "r50"])
@pytest.mark.parametrize("mode", ["eval_frozen", "train_pass1"])
def test_whole_model_x_grad(arch, mode, no_dropout, monkeypatch):
    """x.grad of the drop-in model against the CPU port (same weights, the oracle's op sequence) under autograd.
    The port runs in fp32 like the reference.

    (1) The whole x.grad: the criteria test_hot_path_against_reference_model applies to g_feat (relative L2 < 1e-2,
    every element within 2e-3 relative + 2 % of the maximum), since x.grad passes the same |.| kinks.  Exception: R50
    in train mode at the fixture's R=64, whose backbone BatchNorms normalise over 16 values per channel: there the
    backbone-only x.grad already differs from the port's by ~4e-2 (measured on a B200), so that case is held to 6e-2,
    the floor test_full_model_against_reference uses for the same conditioning.
    (2) The routes this feature adds: delta = x.grad - (x.grad with x detached at the error maps and the
    reconstruction tail), computed the same way on both sides.  The backbone's arithmetic is identical in the two runs
    of one implementation, so its noise cancels in delta; ours must match the port's to 5 % in relative L2.  Without the
    new routes delta is zero and this fails."""
    from unidefense_b200 import ops
    fix = torch.load(os.path.join(GOLDEN, f"full_{arch}.pt"), weights_only=False)
    model, cpu = _models(arch)
    train = mode == "train_pass1"
    for m in (model, cpu):
        m.train(train)
        if not train:
            m.requires_grad_(False)             # the attack setting: only x requires a gradient
    x = P.tensor_for(f"in:full_x_{arch}", (fix["N"], 3, fix["R"], fix["R"]), "unit")
    labels = fix["labels"]
    states = [{k: v.clone() for k, v in m.state_dict().items()} for m in (model, cpu)]

    def run():
        model.load_state_dict(states[0])        # same BatchNorm running stats for every call
        cpu.load_state_dict(states[1])
        xc = x.cuda().requires_grad_()
        ours = torch.autograd.grad(_objective(model(xc), labels.cuda(), train, ops.cross_entropy, ops.triplet_loss),
                                   xc)[0].cpu()
        xr = x.clone().requires_grad_()
        ref = torch.autograd.grad(_objective(cpu(xr), labels, train, F.cross_entropy, O.aw_triplet_loss), xr)[0]
        return ours, ref

    got, want = run()
    err = _rel2(got, want)
    frac_bad = float(((got - want).abs() > 2e-3 * want.abs() + 2e-2 * float(want.abs().max())).float().mean())

    prep, tail, oprep, otail = ops.attn_prep, ops.recon_tail, O.attention_prep, O.recon_tail
    monkeypatch.setattr(ops, "attn_prep", lambda p, xx, s, n="ortho": prep(p, xx.detach(), s, n))
    monkeypatch.setattr(ops, "recon_tail", lambda d, xx, n="ortho": tail(d, xx.detach(), n))
    monkeypatch.setattr(O, "attention_prep", lambda p, xx, s, n="ortho": oprep(p, xx.detach(), s, n))
    monkeypatch.setattr(O, "recon_tail", lambda d, xx, n="ortho": otail(d, xx.detach(), n))
    got_bb, want_bb = run()
    d_got, d_want = got - got_bb, want - want_bb
    d_err = _rel2(d_got, d_want)
    share = float(d_want.norm() / want.norm())
    print(f"{arch} {mode}: x.grad rel. L2 vs CPU port {err:.2e}; new routes: {share:.2e} of |x.grad|, "
          f"ours vs port rel. L2 {d_err:.2e}")
    assert err < (6e-2 if (arch, mode) == ("r50", "train_pass1") else 1e-2), f"x.grad: relative L2 error {err:.3e}"
    if (arch, mode) != ("r50", "train_pass1"):
        assert frac_bad == 0.0, f"x.grad: {frac_bad:.3%} of elements off by more than 2 % of the maximum"
    assert share > 1e-4, "the error-map / reconstruction routes do not reach x in the port"
    assert d_err < 5e-2, f"error-map / reconstruction contribution to x.grad: relative L2 error {d_err:.3e}"
