"""Attribution maps and faithfulness on the GPU: ud_attrib_step, ud_rank_desc and ud_attrib_mask against the torch
compositions of oracle/explain.py, and unidefense_b200.explain's graph-replayed IntegratedGradients, SmoothGrad and
Faithfulness against eager loops that run torch autograd at the same points."""
import os

import numpy as np
import pytest
import torch

import procedural as P
from oracle import explain as E

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LO, HI = -1.0, 1.0
S = 5            # path points of the step-kernel tests


def _ulp(x):
    a = x.abs()
    return torch.nextafter(a, torch.full_like(a, float("inf"))) - a


def _buf(t, offset):
    """A copy of t whose storage starts `offset` floats past an allocation (offset 1: off its 16-byte alignment)."""
    b = torch.empty(t.numel() + offset, device="cuda")[offset:].view_as(t)
    return b.copy_(t)


def _step_state(N, R, seed, offset=0):
    g = torch.Generator().manual_seed(seed)
    s = dict(x=torch.rand(N, 3, R, R, generator=g) * 2 - 1, b=torch.rand(N, 3, R, R, generator=g) * 0.5 - 1,
             g=torch.randn(N, 3, R, R, generator=g), acc=torch.randn(N, 3, R, R, generator=g) * 0.1)
    return {k: _buf(v.cuda(), offset) for k, v in s.items()}


def _tables(method):
    alpha, w = E.ig_tables(S - 1) if method == "ig" else E.smoothgrad_tables(S)
    return (torch.tensor(alpha, dtype=torch.float32, device="cuda"), torch.tensor(w, dtype=torch.float32, device="cuda"))


def _call(s, method, k, tensor_base, start=False, offset=0, sigma=0.3, seed=1234, ids=None):
    """One ud_attrib_step at step k on copies of s; returns acc, p, attr, map."""
    from unidefense_b200 import ops
    x = s["x"]
    acc, p, attr = _buf(s["acc"], offset), _buf(torch.zeros_like(x), offset), _buf(torch.zeros_like(x), offset)
    amap = torch.full(x[:, 0].shape, -7.0, device="cuda")
    alpha, w = _tables(method)
    kt = torch.tensor([k], dtype=torch.int32, device="cuda")
    base = s["b"] if (tensor_base and method == "ig") else (-0.75 if method == "ig" else 0.0)
    sg = method == "smoothgrad"
    ops.attrib_step(x, base, None if start else s["g"], acc, p, attr, amap, kt, alpha, w, method,
                    torch.tensor([sigma], device="cuda") if sg else None, ids,
                    torch.tensor([seed], dtype=torch.int64, device="cuda") if sg else None)
    assert int(kt) == k                                        # the counter is read, never written
    return dict(acc=acc, p=p, attr=attr, map=amap)


def _sg_points(x, k, sigma, seed, ids):
    """fp64 SmoothGrad point k of every sample: x + sigma*eps_k (oracle normals)."""
    P_ = x[0].numel()
    z = np.stack([E.normals(P_, int(i), seed, k) for i in ids])
    return x.double() + sigma * torch.from_numpy(z).to(x.device).view_as(x), torch.from_numpy(z).to(x.device).view_as(x)


# bound for the noisy points: the fp32 Box-Muller (logf / log1pf, sqrtf, sincospif) against fp64, times sigma, plus the
# two fp32 roundings of x + sigma*eps
def _check_sg_points(p, x, k, sigma, seed, ids):
    want, z = _sg_points(x, k, sigma, seed, ids)
    err = (p.double() - want).abs()
    bound = 2 * _ulp(want.float()).double() + sigma * 2e-6 * (z.abs() + 1)
    assert bool((err <= bound).all()), float((err - bound).max())


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["ig", "smoothgrad"])
@pytest.mark.parametrize("N", [1, 4, 32])
@pytest.mark.parametrize("R", [64, 299, 380])
def test_step_kernel_vs_oracle(R, N, method):
    s = _step_state(N, R, seed=R + N)
    x, b, g, acc0 = s["x"], s["b"], s["g"], s["acc"]
    alpha, w = _tables(method)
    sigma, seed = 0.3, 1234
    ids = list(range(N))
    for tensor_base in ((True, False) if method == "ig" else (False,)):
        bb = b if (tensor_base and method == "ig") else torch.full_like(x, -0.75 if method == "ig" else 0.0)
        # start: acc = 0, p = p_k
        out = _call(s, method, 0, tensor_base, start=True)
        assert torch.equal(out["acc"], torch.zeros_like(x))
        if method == "ig":
            assert torch.equal(out["p"], E.path_point(x, bb, float(alpha[0])))
        else:
            _check_sg_points(out["p"], x, 0, sigma, seed, ids)
        # a middle step: acc += w_k g, p = p_{k+1}
        k = 1
        out = _call(s, method, k, tensor_base)
        want_acc = E.accumulate(acc0, float(w[k]), g)
        assert torch.equal(out["acc"], want_acc), "the accumulation is not bit-identical to the torch composition"
        if method == "ig":
            assert torch.equal(out["p"], E.path_point(x, bb, float(alpha[k + 1]))), "IG point is not bit-identical"
        else:
            _check_sg_points(out["p"], x, k + 1, sigma, seed, ids)
        assert torch.equal(out["map"], torch.full_like(out["map"], -7.0))          # the map waits for the last step
        # the last step: attr and map
        out = _call(s, method, S - 1, tensor_base)
        acc = E.accumulate(acc0, float(w[S - 1]), g)
        want_attr = (x - bb) * acc if method == "ig" else acc
        assert torch.equal(out["attr"], want_attr)
        a = out["attr"].abs()
        assert torch.equal(out["map"], (a[:, 0] + a[:, 1]) + a[:, 2])
        again = _call(s, method, S - 1, tensor_base)
        for key in ("attr", "map"):
            assert torch.equal(out[key], again[key]), key
    # out-of-range steps do nothing
    out = _call(s, method, S, False)
    assert torch.equal(out["p"], torch.zeros_like(x)) and torch.equal(out["acc"], acc0)


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["ig", "smoothgrad"])
def test_step_kernel_unaligned_views(method):
    """Tensors off their 16-byte alignment take the scalar loads; arithmetic and noise are the same, bit for bit."""
    a_s, u_s = _step_state(4, 299, seed=3), _step_state(4, 299, seed=3, offset=1)
    for k, start in ((0, True), (1, False), (S - 1, False)):
        a = _call(a_s, method, k, True, start=start)
        u = _call(u_s, method, k, True, start=start, offset=1)
        for key in ("acc", "p", "attr", "map"):
            assert torch.equal(a[key], u[key]), (k, key)


@pytest.mark.gpu
def test_smoothgrad_noise_is_keyed_by_id():
    s = _step_state(4, 64, seed=5)
    ids = torch.tensor([7, 3, 2 ** 40 + 1, -5], dtype=torch.int64, device="cuda")
    full = _call(s, "smoothgrad", 2, False, start=True, ids=ids)
    _check_sg_points(full["p"], s["x"], 2, 0.3, 1234, [7, 3, 2 ** 40 + 1, -5])
    one = _call({k: v[2:3].contiguous() for k, v in s.items()}, "smoothgrad", 2, False, start=True, ids=ids[2:3])
    assert torch.equal(one["p"], full["p"][2:3])


def _torch_rank(m):
    order = torch.sort(-m.flatten(1), dim=1, stable=True).indices
    rank = torch.empty_like(order)
    rank.scatter_(1, order, torch.arange(order.shape[1], device=m.device).expand_as(order))
    return rank.view_as(m).int()


@pytest.mark.gpu
@pytest.mark.parametrize("R", [64, 299, 380, 1024])
def test_rank_desc_equals_stable_torch_sort(R):
    from unidefense_b200 import ops
    g = torch.Generator().manual_seed(R)
    maps = {"random": torch.rand(2, R, R, generator=g),
            "equal": torch.full((2, R, R), 0.25),
            "8bit": torch.round(torch.rand(2, R, R, generator=g) * 255) / 255}
    m = torch.randn(2, R, R, generator=g).abs()
    m.view(2, -1)[0, ::97] = float("nan")
    m.view(2, -1)[1, :3] = torch.tensor([float("inf"), 0.0, -0.0])
    maps["nan"] = m
    for name, mp in maps.items():
        got = ops.rank_desc(mp.cuda())
        assert torch.equal(got, _torch_rank(mp.cuda())), name
        if R <= 299:
            assert np.array_equal(got.cpu().numpy(), E.rank_desc(mp.numpy())), name


@pytest.mark.gpu
@pytest.mark.parametrize("tensor_base", [True, False])
def test_attrib_mask_is_exact(tensor_base):
    from unidefense_b200 import ops
    N, R, K = 3, 97, 7
    s = _step_state(N, R, seed=9)
    x = s["x"]
    b = s["b"] if tensor_base else torch.full_like(x, -1.0)
    rank = ops.rank_desc(torch.rand(N, R, R, device="cuda"))
    t = torch.tensor(E.thresholds(K, R * R), dtype=torch.int32, device="cuda")
    y = torch.empty_like(x)
    for j in (0, 1, 4, K):
        for ins in (False, True):
            ops.attrib_mask(x, b if tensor_base else -1.0, rank, t, torch.tensor([j], dtype=torch.int32, device="cuda"),
                            y, ins)
            assert torch.equal(y, E.masked(x, b, rank, int(t[j]), ins)), (j, ins)


# ---------------------------------------------------------------------------------------------- end to end
CTOR = {"eb4": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2, drop_rate=0.0, drop_connect_rate=0.0)),
        "eb4_1": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=1, drop_rate=0.0, drop_connect_rate=0.0)),
        "r18": ("UDR18", dict(num_classes=2, drop_rate=0.0)),
        "r50": ("UDR50", dict(extractor="resnet50", num_classes=2, drop_rate=0.0))}


def _model(arch):
    from unidefense_b200.model import load_model
    name, kw = CTOR[arch]
    model = load_model(name)(**kw)
    P.fill_state_dict_(model, salt=5)
    return model.cuda().eval()


def _inputs(arch):
    a = arch.split("_")[0]
    fix = torch.load(os.path.join(GOLDEN, f"full_{a}.pt"), weights_only=False)
    x = P.tensor_for(f"in:full_x_{a}", (fix["N"], 3, fix["R"], fix["R"]), "unit").cuda()
    return x, fix["labels"].cuda()


def _grad(model, p, target):
    xin = p.detach().requires_grad_()
    f = E.objective(model(xin)["cls_out"].float(), target)
    g, = torch.autograd.grad(f.sum(), xin)
    return f.detach(), g


def _rel(got, want):
    return float((got.double() - want.double()).norm() / want.double().norm().clamp(min=1e-30))



@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["eb4", "eb4_1", "r18", "r50"])
def test_integrated_gradients_equals_the_eager_loop(arch):
    from unidefense_b200.explain import IntegratedGradients
    model = _model(arch)
    x, _ = _inputs(arch)
    m = 4
    b = torch.full_like(x, LO)
    r = IntegratedGradients(model, steps=m)(x)
    with torch.no_grad():
        logits = model(x)["cls_out"].float()
    target = E.predicted(logits)
    assert torch.equal(r["target"], target)
    alpha, w = E.ig_tables(m)
    acc = torch.zeros_like(x)
    f_b = None
    for k in range(m + 1):
        f, g = _grad(model, E.path_point(x, b, float(np.float32(alpha[k]))), target)
        f_b = f if k == 0 else f_b
        acc = E.accumulate(acc, float(np.float32(w[k])), g)
    attr = (x - b) * acc
    rel = _rel(r["attr"], attr)
    assert rel <= 1e-5, rel
    torch.testing.assert_close(r["f_x"], E.objective(logits, target), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(r["f_baseline"], f_b, rtol=1e-5, atol=1e-6)
    want_delta = attr.flatten(1).double().sum(1) - (r["f_x"].double() - r["f_baseline"].double())
    torch.testing.assert_close(r["delta"], want_delta, rtol=1e-4, atol=1e-5)
    print(f"IG {arch}: normwise rel {rel:.3g}, bit-identical {torch.equal(r['attr'], attr)}")


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["eb4", "eb4_1", "r18", "r50"])
def test_smoothgrad_equals_the_eager_loop(arch):
    """The eager loop takes the gradient at the points the kernel emits (start calls at each k)."""
    from unidefense_b200 import ops
    from unidefense_b200.explain import SmoothGrad
    model = _model(arch)
    x, labels = _inputs(arch)
    draws, noise, seed = 3, 0.1, 77
    r = SmoothGrad(model, draws=draws, noise=noise)(x, labels=labels, seed=seed)
    assert torch.equal(r["target"], labels)
    alpha, w = E.smoothgrad_tables(draws)
    at, wt = (torch.tensor(v, dtype=torch.float32, device="cuda") for v in (alpha, w))
    sigma = torch.tensor([noise * (HI - LO)], device="cuda")
    acc = torch.zeros_like(x)
    for k in range(draws):
        p = torch.empty_like(x)
        ops.attrib_step(x, 0.0, None, torch.empty_like(x), p, torch.empty_like(x), torch.empty_like(x[:, 0]),
                        torch.tensor([k], dtype=torch.int32, device="cuda"), at, wt, "smoothgrad", sigma, None,
                        torch.tensor([seed], dtype=torch.int64, device="cuda"))
        _check_sg_points(p, x, k, float(sigma), seed, range(x.shape[0]))
        acc = E.accumulate(acc, float(wt[k]), _grad(model, p, labels)[1])
    rel = _rel(r["attr"], acc)
    assert rel <= 1e-5, rel
    a = acc.abs()
    assert _rel(r["map"], (a[:, 0] + a[:, 1]) + a[:, 2]) <= 1e-5
    print(f"SmoothGrad {arch}: normwise rel {rel:.3g}, bit-identical {torch.equal(r['attr'], acc)}")


@pytest.mark.gpu
def test_vanilla_gradient_is_smoothgrad_without_noise():
    from unidefense_b200.explain import SmoothGrad
    model = _model("r18")
    x, labels = _inputs("r18")
    r = SmoothGrad(model, draws=1, noise=0.0)(x, labels=labels)
    _, g = _grad(model, x, labels)
    assert _rel(r["attr"], g) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["eb4", "eb4_1", "r18", "r50"])
def test_faithfulness_equals_the_eager_loop(arch):
    from unidefense_b200.explain import Faithfulness
    model = _model(arch)
    x, labels = _inputs(arch)
    N, _, H, W = x.shape
    K = 5
    amap = torch.rand(N, H, W, device="cuda")
    b = torch.full_like(x, LO)
    c = Faithfulness(model, points=K)(x, amap, labels=labels)
    rank = _torch_rank(amap)
    want = {"deletion": [], "insertion": []}
    with torch.no_grad():
        for t in E.thresholds(K, H * W):
            for name, ins in (("deletion", False), ("insertion", True)):
                logits = model(E.masked(x, b, rank, t, ins))["cls_out"].float()
                want[name].append(E.objective(logits, labels).exp())
    for name in ("deletion", "insertion"):
        wnt = torch.stack(want[name], 1)
        rel = _rel(c[name], wnt)
        assert rel <= 1e-5, (name, rel)
        torch.testing.assert_close(c[f"{name}_auc"], E.auc(wnt), rtol=1e-5, atol=1e-6)
    # the endpoints: j = 0 deletes nothing, j = K deletes every pixel
    with torch.no_grad():
        p_x = E.objective(model(x)["cls_out"].float(), labels).exp()
        p_b = E.objective(model(b)["cls_out"].float(), labels).exp()
    torch.testing.assert_close(c["deletion"][:, 0], p_x, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(c["deletion"][:, K], p_b, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(c["insertion"][:, 0], p_b, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(c["insertion"][:, K], p_x, rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_completeness_error_falls_with_steps():
    from unidefense_b200.explain import IntegratedGradients
    model = _model("r18")
    x, _ = _inputs("r18")
    d8 = IntegratedGradients(model, steps=8)(x)["delta"].abs().mean()
    d64 = IntegratedGradients(model, steps=64)(x)["delta"].abs().mean()
    print(f"UDR18 mean |delta|: m=8 {float(d8):.4g}, m=64 {float(d64):.4g}")
    assert float(d64) < float(d8)


@pytest.mark.gpu
def test_new_inputs_replay_without_a_new_capture():
    from unidefense_b200 import _lib
    from unidefense_b200.explain import Faithfulness, IntegratedGradients, SmoothGrad
    model = _model("eb4")
    x, labels = _inputs("eb4")
    lib = _lib.lib()
    ig, sg, fa = IntegratedGradients(model, steps=6), SmoothGrad(model, draws=4), Faithfulness(model, points=4)
    r = ig(x)
    sg(x)
    fa(x, r["map"])
    x2 = torch.flip(x, dims=[3]).contiguous()
    blur = torch.nn.functional.avg_pool2d(x, 5, 1, 2)
    n0 = lib.ud_launch_count()
    r2 = ig(x2, labels=labels, baseline=blur)
    r3 = ig(x, baseline=0.0)
    sg(x2, seed=5)
    fa(x2, r2["map"], baseline=blur)
    moved = lib.ud_launch_count() - n0
    assert moved <= 2, f"{moved} library launches outside the replayed graphs"     # the rank sort of Faithfulness
    assert len(ig._graphs) == len(sg._graphs) == len(fa._graphs) == 1
    assert not torch.equal(r2["attr"], r["attr"]) and not torch.equal(r3["attr"], r["attr"])
    again = ig(x2, labels=labels, baseline=blur)
    assert torch.equal(again["attr"], r2["attr"]) and torch.equal(again["map"], r2["map"])


@pytest.mark.gpu
def test_bf16_autocast_runs():
    from unidefense_b200.explain import Faithfulness, IntegratedGradients, SmoothGrad
    model = _model("eb4")
    x, _ = _inputs("eb4")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        r = IntegratedGradients(model, steps=4)(x)
        s = SmoothGrad(model, draws=2)(x)
        c = Faithfulness(model, points=4)(x, r["map"])
    for t in (r["attr"], r["map"], r["delta"], s["attr"], c["deletion"], c["insertion_auc"]):
        assert bool(torch.isfinite(t).all())
    assert r["attr"].dtype == torch.float32


@pytest.mark.gpu
def test_rejections():
    from unidefense_b200.explain import Faithfulness, IntegratedGradients, SmoothGrad
    model = _model("r18")
    x, labels = _inputs("r18")
    for bad in (dict(steps=0),):
        with pytest.raises(ValueError, match="steps"):
            IntegratedGradients(model, **bad)
    with pytest.raises(ValueError, match="draws"):
        SmoothGrad(model, draws=0)
    with pytest.raises(ValueError, match="noise must be >= 0"):
        SmoothGrad(model, noise=-0.1)
    with pytest.raises(ValueError, match="points"):
        Faithfulness(model, points=0)
    ig, sg, fa = IntegratedGradients(model, steps=2), SmoothGrad(model, draws=1), Faithfulness(model, points=2)
    amap = torch.rand(x.shape[0], *x.shape[2:], device="cuda")
    with pytest.raises(RuntimeError, match="train mode"):
        IntegratedGradients(model.train(), steps=1)(x)
    model.eval()
    for call in (lambda v: ig(v), lambda v: sg(v), lambda v: fa(v, amap)):
        with pytest.raises(RuntimeError, match="CUDA fp32"):
            call(x.cpu())
        with pytest.raises(RuntimeError, match="CUDA fp32"):
            call(x.double())
        with pytest.raises(ValueError, match=r"\[N, C, H, W\]"):
            call(x[0])
    with pytest.raises(ValueError, match="labels for a batch"):
        ig(x, labels=labels[:2])
    with pytest.raises(ValueError, match="baseline"):
        ig(x, baseline=x[:, :1])
    with pytest.raises(ValueError, match="ids"):
        sg(x, ids=torch.arange(2, device="cuda"))
    with pytest.raises(ValueError, match="seed"):
        sg(x, seed=-1)
    with pytest.raises(ValueError, match="map must be"):
        fa(x, amap[:, :-1])
    with pytest.raises(RuntimeError, match="map must be an fp32"):
        fa(x, amap.double())
    if torch.cuda.device_count() > 1:
        with pytest.raises(RuntimeError, match="current device"):
            ig(x.to("cuda:1"))
