"""PGD / FGSM robustness evaluation: ud_attack_step against the torch composition of oracle/attack.py, and the graph-
replayed attack (unidefense_b200.attack.PGD) against an eager loop written with the oracle and torch.autograd.grad."""
import math
import os

import pytest
import torch
import torch.nn.functional as F

import procedural as P
from oracle import attack as A

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LO, HI = -1.0, 1.0


def _ulp(x):
    a = x.abs()
    return torch.nextafter(a, torch.full_like(a, math.inf)) - a


def _within_linf_ball(x_adv, x0, eps):
    """|x_adv - x0| <= eps + ulp: x_adv = fl(x0 + delta) with |delta| <= eps rounds once, at the magnitude of the larger
    of x0 and x_adv (ulp(x0) alone is too small where |x0| < |x_adv|).  The difference is taken in fp64."""
    d = (x_adv.double() - x0.double()).abs()
    return bool((d <= eps.double().view(-1, *([1] * (x0.dim() - 1))) + _ulp(torch.maximum(x0.abs(), x_adv.abs()))).all())


def _state(N, per_sample, seed, offset=0, norm="linf"):
    """x0 in [-1, 1] with pixels on the range boundary, an iterate inside the ball, a gradient with zeros, and losses
    that improve, tie, are NaN or are worse.  offset > 0 puts every tensor off its 16-byte alignment.  L2 radii are
    0.01-0.03 per element (times sqrt(per_sample)): far above fp32 resolution, so that the stored fp32 x_adv - x0 can be
    held to 1e-5 relative."""
    g = torch.Generator().manual_seed(seed)

    def img(t):
        buf = torch.empty(N * per_sample + offset, device="cuda")
        v = buf[offset:].view(N, per_sample)
        v.copy_(t)
        return v

    x0 = torch.rand(N, per_sample, generator=g) * 2 - 1
    x0[:, :5] = HI
    x0[:, 5:10] = LO
    eps = torch.rand(N, generator=g) * 0.2 + 0.01
    if norm == "l2":
        eps = (torch.rand(N, generator=g) + 0.5) * 0.02 * math.sqrt(per_sample)
    x_adv = torch.clamp(x0 + (torch.rand(N, per_sample, generator=g) * 2 - 1) * eps[:, None], LO, HI)
    grad = torch.randn(N, per_sample, generator=g)
    grad[:, 10:20] = 0.0
    alpha = eps * 0.7
    kinds = torch.arange(N) % 4                  # 0 improved, 1 tied, 2 NaN loss, 3 worse
    best = torch.randn(N, generator=g)
    loss = torch.where(kinds == 0, best + 0.5, torch.where(kinds == 1, best, best - 0.5))
    loss[kinds == 2] = math.nan
    x_best = torch.randn(N, per_sample, generator=g)
    return dict(x0=img(x0), x_adv=img(x_adv), g=img(grad), loss=loss.cuda(), best_loss=best.cuda(), x_best=img(x_best),
                eps=eps.cuda(), alpha=alpha.cuda())


def _run(s, norm, step=True):
    from unidefense_b200 import ops
    out = {}
    for k, v in s.items():          # copies at the same offset from a 16-byte boundary as the inputs
        o = torch.empty(v.numel() + v.storage_offset(), device="cuda")[v.storage_offset():].view_as(v)
        out[k] = o.copy_(v)
    ops.attack_step(out["x0"], out["x_adv"], out["g"] if step else None, out["loss"], out["best_loss"], out["x_best"],
                    out["eps"], out["alpha"], LO, HI, norm)
    return out


def _check_select(s, out):
    nb, nx, imp = A.select(s["loss"], s["best_loss"], s["x_adv"], s["x_best"])
    assert torch.equal(out["best_loss"], nb)
    assert torch.equal(out["x_best"], nx)             # improved rows copy x_adv before the step; the rest keep bits
    assert torch.equal(out["x_best"][~imp], s["x_best"][~imp])
    return imp


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ["linf", "l2"])
@pytest.mark.parametrize("N", [1, 4, 32])
@pytest.mark.parametrize("per_sample", [3 * 64 * 64, 3 * 299 * 299, 3 * 380 * 380])
def test_step_kernel_vs_oracle(per_sample, N, norm):
    s = _state(N, per_sample, seed=per_sample + N, norm=norm)
    out = _run(s, norm)
    imp = _check_select(s, out)
    if N >= 4:
        assert imp.tolist()[:4] == [True, False, False, False]
    x0 = s["x0"]
    if norm == "linf":
        want = A.linf_step(x0, s["x_adv"], s["g"], s["eps"], s["alpha"], LO, HI)
        assert torch.equal(out["x_adv"], want), "L-inf step is not bit-identical to the torch composition"
    else:
        want = A.l2_step(x0.double(), s["x_adv"].double(), s["g"].double(), s["eps"].double(), s["alpha"].double(),
                         LO, HI)
        d_got, d_want = (out["x_adv"].double() - x0.double()), (want - x0.double())
        rel = (d_got - d_want).norm(dim=1) / d_want.norm(dim=1)
        assert float(rel.max()) < 1e-5, rel
    # constraints of the output
    if norm == "linf":
        assert _within_linf_ball(out["x_adv"], x0, s["eps"])
    else:
        r = (out["x_adv"].double() - x0.double()).norm(dim=1)
        assert bool((r <= s["eps"].double() * (1 + 1e-6)).all()), (r / s["eps"] - 1).max()
    assert float(out["x_adv"].min()) >= LO and float(out["x_adv"].max()) <= HI
    # bitwise reproducible, including the L2 norms
    again = _run(s, norm)
    for k in ("x_adv", "x_best", "best_loss"):
        assert torch.equal(out[k], again[k]), k
    # select only: x_adv untouched
    sel = _run(s, norm, step=False)
    _check_select(s, sel)
    assert torch.equal(sel["x_adv"], s["x_adv"])


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ["linf", "l2"])
def test_step_kernel_unaligned_tensors(norm):
    """Tensors off their 16-byte alignment take the scalar loads; the arithmetic is the same."""
    per_sample = 3 * 299 * 299
    a = _run(_state(4, per_sample, seed=7, offset=1, norm=norm), norm)
    b = _run(_state(4, per_sample, seed=7, norm=norm), norm)
    for k in ("x_adv", "x_best", "best_loss"):
        if norm == "linf" or k != "x_adv":
            assert torch.equal(a[k], b[k]), k
        else:       # the L2 partial sums run over other index ranges
            torch.testing.assert_close(a[k], b[k], rtol=0, atol=1e-6)


# ---------------------------------------------------------------------------------------------- end to end
CTOR = {"eb4": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2, drop_rate=0.0, drop_connect_rate=0.0)),
        "r18": ("UDR18", dict(num_classes=2, drop_rate=0.0)),
        "r50": ("UDR50", dict(extractor="resnet50", num_classes=2, drop_rate=0.0))}


def _model(arch, **over):
    from unidefense_b200.model import load_model
    name, kw = CTOR[arch]
    model = load_model(name)(**{**kw, **over})
    P.fill_state_dict_(model, salt=5)
    return model.cuda().eval()


def _inputs(arch):
    fix = torch.load(os.path.join(GOLDEN, f"full_{arch}.pt"), weights_only=False)
    x = P.tensor_for(f"in:full_x_{arch}", (fix["N"], 3, fix["R"], fix["R"]), "unit").cuda()
    return x, fix["labels"].cuda()


def _per_sample_loss(logits, labels):
    logits = logits.float()
    if logits.shape[1] == 1:
        return F.binary_cross_entropy_with_logits(logits[:, 0], labels.float(), reduction="none")
    return F.cross_entropy(logits, labels, reduction="none")


def _eager_pgd(model, x0, labels, eps, alpha, steps, norm):
    """The hand-written loop: forward, autograd.grad, select, step; one more forward scores the last iterate."""
    N = x0.shape[0]
    e, a = torch.full((N,), eps, device="cuda"), torch.full((N,), alpha, device="cuda")
    step = A.linf_step if norm == "linf" else A.l2_step
    x_adv, x_best = x0.clone(), x0.clone()
    best = torch.full((N,), -math.inf, device="cuda")
    for _ in range(steps):
        xin = x_adv.detach().requires_grad_()
        loss = _per_sample_loss(model(xin)["cls_out"], labels)
        g, = torch.autograd.grad(loss.sum(), xin)
        best, x_best, _ = A.select(loss.detach(), best, x_adv, x_best)
        x_adv = step(x0, x_adv, g, e, a, LO, HI)
    with torch.no_grad():
        loss = _per_sample_loss(model(x_adv)["cls_out"], labels)
    best, x_best, _ = A.select(loss, best, x_adv, x_best)
    return x_best, best


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["eb4", "r18", "r50"])
@pytest.mark.parametrize("norm,steps", [("linf", 3), ("l2", 1), ("l2", 3)])
def test_pgd_equals_the_eager_loop(arch, norm, steps):
    """L-inf: bit for bit.  L2: the kernel's and torch's norms add in different orders, so the iterates differ in the
    last bits; after one step delta agrees to 1e-4.  Later steps take the gradient at those slightly different points,
    and the ReLU / max-pool kinks of the backbones amplify the difference (measured on a B200: up to 1.2e-3 relative
    after three steps of UDR50), so three steps are held to 1e-2 and to the same best loss."""
    from unidefense_b200.attack import PGD
    model = _model(arch)
    x, labels = _inputs(arch)
    eps = 16 / 255 if norm == "linf" else 1.0
    res = PGD(model, norm=norm, steps=steps, random_start=False)(x, labels, eps=eps)
    want_x, want_best = _eager_pgd(model, x, labels, eps, 2.5 * eps / steps, steps, norm)
    if norm == "linf":
        assert torch.equal(res["x_adv"], want_x), "graph-replayed L-inf iterates differ from the eager loop"
        torch.testing.assert_close(res["best_loss"], want_best, rtol=1e-5, atol=1e-6)
    else:
        d_got, d_want = (res["x_adv"] - x).flatten(1).double(), (want_x - x).flatten(1).double()
        rel = (d_got - d_want).norm(dim=1) / d_want.norm(dim=1).clamp(min=1e-30)
        assert float(rel.max()) < (1e-4 if steps == 1 else 1e-2), rel
        torch.testing.assert_close(res["best_loss"], want_best, rtol=1e-5 if steps == 1 else 1e-3, atol=1e-6)
    with torch.no_grad():
        logits = model(res["x_adv"])["cls_out"]
    torch.testing.assert_close(res["logits"], logits, rtol=1e-4, atol=1e-5)
    assert res["fooled"].dtype == torch.bool and res["fooled"].shape == labels.shape
    assert bool((res["fooled"] | (logits.argmax(dim=1) == labels)).all())     # a misclassified best iterate fooled


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["eb4", "r18", "r50"])
def test_fgsm_is_the_signed_gradient_step(arch):
    from unidefense_b200.attack import PGD
    model = _model(arch)
    x, labels = _inputs(arch)
    eps = 8 / 255
    res = PGD(model, steps=1, random_start=False)(x, labels, eps=eps, alpha=eps)
    xin = x.clone().requires_grad_()
    loss = _per_sample_loss(model(xin)["cls_out"], labels)
    g, = torch.autograd.grad(loss.sum(), xin)
    fgsm = torch.clamp(x + eps * torch.sign(g), LO, HI)
    with torch.no_grad():
        l_fgsm = _per_sample_loss(model(fgsm)["cls_out"], labels)
    moved = l_fgsm > loss.detach()                  # the best iterate is the FGSM point wherever it raised the loss
    torch.testing.assert_close(res["x_adv"][moved], fgsm[moved], rtol=0, atol=float(_ulp(x).max()))
    assert torch.equal(res["x_adv"][~moved], x[~moved])


@pytest.mark.gpu
def test_bce_objective_of_a_single_logit_model():
    """num_classes == 1 (UDEB4's default) ascends BCE-with-logits; misclassified = (logit > 0) != label."""
    from unidefense_b200.attack import PGD
    model = _model("r18", num_classes=1)
    x, labels = _inputs("r18")
    res = PGD(model, steps=2, random_start=False)(x, labels, eps=16 / 255)
    want_x, want_best = _eager_pgd(model, x, labels, 16 / 255, 2.5 * 16 / 255 / 2, 2, "linf")
    assert torch.equal(res["x_adv"], want_x)
    torch.testing.assert_close(res["best_loss"], want_best, rtol=1e-5, atol=1e-6)
    assert res["logits"].shape == (x.shape[0], 1)


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ["linf", "l2"])
def test_best_tracking_and_restarts(norm):
    from unidefense_b200.attack import PGD
    model = _model("r18")
    x, labels = _inputs("r18")
    eps = 16 / 255 if norm == "linf" else 1.0
    with torch.no_grad():
        first = _per_sample_loss(model(x)["cls_out"], labels)
    res = PGD(model, norm=norm, steps=3, random_start=False)(x, labels, eps=eps)
    assert bool((res["best_loss"] >= first).all())
    torch.manual_seed(11)
    one = PGD(model, norm=norm, steps=3, restarts=1)(x, labels, eps=eps)
    torch.manual_seed(11)
    two = PGD(model, norm=norm, steps=3, restarts=2)(x, labels, eps=eps)
    assert bool((two["best_loss"] >= one["best_loss"]).all()), (one["best_loss"], two["best_loss"])
    d = (two["x_adv"] - x).flatten(1)
    r = d.abs().amax(1) if norm == "linf" else d.double().norm(dim=1)
    assert bool((r <= eps * (1 + 1e-6) + 1e-6).all())


@pytest.mark.gpu
def test_iterations_replay_a_captured_graph():
    from unidefense_b200 import _lib
    from unidefense_b200.attack import PGD
    model = _model("eb4")
    x, labels = _inputs("eb4")
    atk = PGD(model, steps=10)
    atk(x, labels, eps=8 / 255)                     # captures
    lib = _lib.lib()
    n0 = lib.ud_launch_count()
    atk(x, labels, eps=8 / 255)
    atk(x, labels, eps=16 / 255)                    # another eps: same graphs
    moved = lib.ud_launch_count() - n0
    assert moved <= 4, f"{moved} library launches for two 10-step attacks: the iterations are not replayed"
    assert len(atk._graphs) == 1
    with torch.autocast("cuda", dtype=torch.bfloat16):
        res = atk(x, labels, eps=16 / 255)          # a new autocast state is a new capture
    assert len(atk._graphs) == 2
    d = (res["x_adv"] - x).abs()
    assert _within_linf_ball(res["x_adv"], x, torch.full((x.shape[0],), 16 / 255, device="cuda"))
    assert bool(torch.isfinite(res["best_loss"]).all())


@pytest.mark.gpu
def test_rejections():
    from unidefense_b200 import _lib
    from unidefense_b200.attack import PGD
    model = _model("r18")
    x, labels = _inputs("r18")
    atk = PGD(model, steps=1)
    with pytest.raises(RuntimeError, match="train mode"):
        PGD(model.train(), steps=1)(x, labels)
    model.eval()
    with pytest.raises(RuntimeError, match="CUDA fp32"):
        atk(x.cpu(), labels)
    with pytest.raises(RuntimeError, match="CUDA fp32"):
        atk(x.double(), labels)
    with pytest.raises(ValueError, match="eps must be >= 0"):
        atk(x, labels, eps=-0.1)
    with pytest.raises(ValueError, match="labels for a batch"):
        atk(x, labels[:2])
    with pytest.raises(ValueError, match="norm must be"):
        PGD(model, norm="l1")
    s = _state(2, 3 * 64 * 64, seed=1)
    lib = _lib.lib()
    nws = lib.ud_attack_workspace_bytes(2, 3 * 64 * 64)
    ws = torch.empty(nws - 4, dtype=torch.uint8, device="cuda")
    rc = lib.ud_attack_step(*(s[k].data_ptr() for k in ("x0", "x_adv", "g", "loss", "best_loss", "x_best", "eps",
                                                         "alpha")), LO, HI, 0, 2, 3 * 64 * 64, ws.data_ptr(),
                            ws.numel(), torch.cuda.current_stream().cuda_stream)
    assert rc == -4 and b"workspace" in lib.ud_last_error()
