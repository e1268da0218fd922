"""Fourier heat maps on the GPU: ud_fourier_perturb against the fp64 oracle of oracle/fourier.py (values, clamp,
spectrum and norm), its keying, unaligned views and reproducibility, and unidefense_b200.fourier's graph-replayed
FourierHeatMap against an eager loop of perturb + forward + scores."""
import math

import numpy as np
import pytest
import torch

import procedural as P
from oracle import corrupt as C
from oracle import fourier as FO

LO, HI = -1.0, 1.0
SEED = 0x0123456789ABCDEF


def _ulp(x):
    a = x.abs()
    return torch.nextafter(a, torch.full_like(a, float("inf"))) - a


def _buf(t, offset):
    """A copy of t whose storage starts `offset` floats past an allocation (offset 1: off its 16-byte alignment)."""
    b = torch.empty(t.numel() + offset, device=t.device)[offset:].view_as(t)
    return b.copy_(t)


def _table(H, W):
    """Canonical pairs: DC, the Nyquist row, column and corner, negative u, and a few others."""
    pts = [(0, 0), (H // 2, 0), (0, W // 2), (H // 2, W // 2), (-5, 3), (-1, 0), (7, W // 3), (H // 3, -2)]
    return sorted({FO.canonical(u, v, H, W) for u, v in pts})


def _i32(v):
    return torch.tensor([v], dtype=torch.int32, device="cuda")


def _perturb(x, table, f, eps, ids=None, seed=SEED, y=None, lo=LO, hi=HI):
    from unidefense_b200 import ops
    y = torch.full_like(x, 7.0) if y is None else y
    ops.fourier_perturb(x, y, torch.tensor(table, dtype=torch.int32, device="cuda").view(-1, 2), _i32(f),
                        torch.tensor([eps], dtype=torch.float32, device="cuda"), ids,
                        torch.tensor([seed - 2 ** 64 if seed >= 2 ** 63 else seed], dtype=torch.int64, device="cuda"),
                        lo, hi)
    return y


# Error bound against the fp64 oracle, per element, with s the kernel's (exact, fp32) step:
#  - t = k/(H*W) is one rounded fp32 division of exact integers; t < 1, so |dt| <= ulp(t)/2 <= 2^-25 and the cosine
#    moves by at most 2*pi*2^-25;
#  - cospif is within 1 ulp, and |c| < 1 away from its exact +-1 points, so that is <= 2^-24; the product s*c rounds
#    once more, <= |s|*2^-24: together |s|*2^-23;
#  - x + s*c rounds once: <= ulp(y)/2; clamping to [lo, hi] cannot increase the error.
# The fp64 oracle's own error (~1e-16 relative) is covered by the 1e-12*|s| slack.
def _bound(got, want, s):
    half_ulp = torch.maximum(_ulp(got), _ulp(want.float())).double() / 2
    return half_ulp + s.abs() * (2 * math.pi * 2.0 ** -25 + 2.0 ** -23 + 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 4, 32])
@pytest.mark.parametrize("H,W", [(64, 64), (299, 299), (380, 380), (45, 67)])
def test_kernel_vs_fp64_oracle(H, W, N):
    g = torch.Generator().manual_seed(H * W + N)
    x = (torch.rand(N, 3, H, W, generator=g) * 2 - 1).cuda()
    table = _table(H, W)
    eps = 0.05 / FO.amplitude(1, 1, H, W)                            # peak 0.05: the clamp acts near +-1
    ids = list(range(100, 100 + N))
    idt = torch.tensor(ids, dtype=torch.int64, device="cuda")
    x_np = x.cpu().numpy()
    clamped = 0
    for fi, (uu, vv) in enumerate(table):
        got = _perturb(x, table, fi, eps, idt)
        want = torch.from_numpy(FO.perturb(x_np, uu, vv, eps, ids, SEED, LO, HI)).cuda()
        s = torch.from_numpy(FO.step(uu, vv, H, W, eps, FO.signs(ids, 3, uu, vv, SEED))).cuda()[:, :, None, None]
        bound = _bound(got, want, s)
        err = (got.double() - want).abs()
        assert bool((err <= bound).all()), ((uu, vv), float((err - bound).max()))
        c = torch.from_numpy(np.cos(2 * np.pi * FO.phase(uu, vv, H, W) / (H * W))).cuda()
        raw = x.double() + s * c
        hi_c, lo_c = raw > HI + bound, raw < LO - bound
        assert bool((got[hi_c] == HI).all()) and bool((got[lo_c] == LO).all()), (uu, vv)
        clamped += int(hi_c.sum() + lo_c.sum())
    assert clamped > 0


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(64, 96), (45, 67), (380, 380)])
def test_gpu_basis_spectrum_and_norm(H, W):
    """With x = 0 and no clamp, (y - x)/(r*eps) is the basis: unit norm per plane, spectrum only at +-(u, v)."""
    N, eps = 2, 1.0
    x = torch.zeros(N, 3, H, W, device="cuda")
    table = _table(H, W)
    for fi, (uu, vv) in enumerate(table):
        y = _perturb(x, table, fi, eps).double().cpu().numpy()
        r = FO.signs([0, 1], 3, uu, vv, SEED)
        d = y / (r[:, :, None, None] * eps)
        norms = np.sqrt((d ** 2).sum((2, 3)))
        assert np.abs(norms - 1).max() < 1e-6, ((uu, vv), norms)
        e = np.abs(np.fft.fft2(d)) ** 2
        keep = np.zeros((H, W), bool)
        keep[uu, vv] = keep[(-uu) % H, (-vv) % W] = True
        leak = e[..., ~keep].sum((-1)) / e.sum((-2, -1))
        assert leak.max() < 1e-12, ((uu, vv), leak.max())


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(64, 64), (45, 67)])
def test_keying_views_and_reproducibility(H, W):
    N = 6
    g = torch.Generator().manual_seed(7)
    x = (torch.rand(N, 3, H, W, generator=g) * 2 - 1).cuda()
    ids = torch.tensor([10, 11, 12, 2 ** 40 + 3, -4, 15], dtype=torch.int64, device="cuda")
    table = _table(H, W)
    fi, eps = 4, 3.0
    full = _perturb(x, table, fi, eps, ids)
    assert torch.equal(full, _perturb(x, table, fi, eps, ids))                       # two calls: bitwise equal
    one = _perturb(x[3:4].contiguous(), table, fi, eps, ids[3:4].contiguous())
    assert torch.equal(one, full[3:4])                                               # no neighbours
    perm = torch.tensor([5, 2, 0, 4, 1, 3], device="cuda")
    assert torch.equal(_perturb(x[perm].contiguous(), table, fi, eps, ids[perm].contiguous()), full[perm])
    rev = table[::-1]
    assert torch.equal(_perturb(x, rev, len(table) - 1 - fi, eps, ids), full)        # table order
    for xo, yo in ((1, 1), (0, 1), (1, 0), (3, 2)):                                  # unaligned views
        got = _perturb(_buf(x, xo), table, fi, eps, ids, y=_buf(torch.zeros_like(x), yo))
        assert torch.equal(got, full), (xo, yo)
    # id 0..N-1 by default
    assert torch.equal(_perturb(x, table, fi, eps), _perturb(x, table, fi, eps, torch.arange(N, device="cuda")))
    # f out of range, or a table entry off the image, writes nothing
    for t, f in ((table, len(table)), (table, -1), ([(H, 0)], 0), ([(0, W)], 0), ([(-1, 0)], 0)):
        assert torch.equal(_perturb(x, t, f, eps, ids), torch.full_like(x, 7.0)), (t, f)


# ---------------------------------------------------------------------------------------------- end to end
CTOR = {"eb4": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2, drop_rate=0.0, drop_connect_rate=0.0)),
        "eb4_1": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=1, drop_rate=0.0, drop_connect_rate=0.0)),
        "r18": ("UDR18", dict(num_classes=2, drop_rate=0.0))}


def _model(arch):
    from unidefense_b200.model import load_model
    name, kw = CTOR[arch]
    model = load_model(name)(**kw)
    P.fill_state_dict_(model, salt=5)
    return model.cuda().eval()


def _batches(R=64, sizes=(5, 7)):
    x = torch.from_numpy(C.test_images(sum(sizes), R, R, seed=1)).cuda()
    labels = torch.tensor([0, 1] * ((sum(sizes) + 1) // 2), device="cuda")[:sum(sizes)]
    out, i = [], 0
    for n in sizes:
        out.append((x[i:i + n], labels[i:i + n]))
        i += n
    return out


def _nan_equal(a, b):
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    return bool(((a == b) | (a.isnan() & b.isnan())).all())


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["r18", "eb4", "eb4_1"])
def test_heat_map_equals_the_eager_loop(arch):
    from unidefense_b200 import corrupt, ops
    from unidefense_b200._evaluator import auc, p_fake
    from unidefense_b200.fourier import FourierHeatMap, grid
    model = _model(arch)
    batches = _batches()
    radius, eps, seed = 2, 2.0, 99
    r = FourierHeatMap(model, eps, radius=radius)(batches, seed=seed)
    u, v, table, index = grid(64, 64, radius, 16)
    assert r["u"].tolist() == u == [-32, -16, 0, 16, 32] and r["v"].tolist() == v == [0, 16, 32]
    assert r["acc"].shape == r["auc"].shape == (5, 3) and r["acc"].dtype == r["auc"].dtype == torch.float64
    assert r["eps"] == eps and r["peak"] == eps * math.sqrt(2 / 64 ** 2)
    freqs = torch.tensor(table, dtype=torch.int32, device="cuda")
    labels = torch.cat([b[1] for b in batches])
    want_acc, want_auc = [], []
    with torch.no_grad():
        for fi in range(len(table)):
            ps, hits, n = [], [], 0
            for x, lab in batches:
                y = torch.empty_like(x)
                ops.fourier_perturb(x, y, freqs, _i32(fi), torch.tensor([eps], device="cuda"),
                                    torch.arange(n, n + x.shape[0], device="cuda"),
                                    torch.tensor([seed], dtype=torch.int64, device="cuda"), LO, HI)
                p, pred = p_fake(model(y)["cls_out"])
                ps.append(p)
                hits.append(pred == lab)
                n += x.shape[0]
            want_acc.append(float(torch.cat(hits).double().mean()))
            want_auc.append(float(auc(torch.cat(ps), labels)))
    for i in range(len(u)):
        for j in range(len(v)):
            k = index[i][j]
            assert float(r["acc"][i, j]) == want_acc[k], (u[i], v[j])
            assert _nan_equal(r["auc"][i, j], want_auc[k]), (u[i], v[j], float(r["auc"][i, j]), want_auc[k])
    for i in range(len(u)):                                     # mirror points: (u, 0) ~ (-u, 0), (u, 32) ~ (-u, 32)
        for j in (0, 2):
            assert float(r["acc"][i, j]) == float(r["acc"][len(u) - 1 - i, j])
            assert _nan_equal(r["auc"][i, j], r["auc"][len(u) - 1 - i, j])
    clean = corrupt.evaluate(model, batches, kinds=())["clean"]
    assert r["clean"]["n"] == clean["n"] == 12 and r["clean"]["acc"] == clean["acc"]
    assert _nan_equal(r["clean"]["auc"], clean["auc"])
    print(f"{arch}: clean {r['clean']}, acc {r['acc'].tolist()}")


@pytest.mark.gpu
def test_new_eps_seed_and_batch_replay_without_a_new_capture():
    from unidefense_b200 import _lib
    from unidefense_b200.fourier import FourierHeatMap
    model = _model("r18")
    (x, lab), = _batches(sizes=(6,))
    hm = FourierHeatMap(model, 4.0, radius=2)
    r0 = hm([(x, lab)], seed=1)
    assert len(hm._graphs) == 1
    lib = _lib.lib()
    n0 = lib.ud_launch_count()
    hm.eps = 12.0
    r1 = hm([(x, lab)], seed=1)
    r2 = hm([(x, lab)], seed=2 ** 64 - 1)
    r3 = hm([(torch.flip(x, dims=[3]).contiguous(), lab, torch.arange(50, 56, device="cuda"))], seed=1)
    assert lib.ud_launch_count() == n0, "library launches outside the replayed graphs"
    assert len(hm._graphs) == 1
    hm.eps = 4.0
    again = hm([(x, lab)], seed=1)
    for key in ("acc", "auc"):
        assert _nan_equal(again[key], r0[key])
    assert r1["peak"] == 3 * r0["peak"] and r1["clean"] == r0["clean"]
    assert r2["clean"] == r0["clean"] and r3["acc"].shape == r0["acc"].shape
    hm([(x[:4], lab[:4])])                                       # a new batch size is a new shape: one more capture
    assert len(hm._graphs) == 2


@pytest.mark.gpu
def test_bf16_autocast_runs():
    from unidefense_b200.fourier import FourierHeatMap
    model = _model("eb4")
    batches = _batches(sizes=(4, 4))
    with torch.autocast("cuda", dtype=torch.bfloat16):
        r = FourierHeatMap(model, 2.0, radius=2)(batches)
    assert r["acc"].shape == (5, 3) and bool(((r["acc"] >= 0) & (r["acc"] <= 1)).all())
    assert bool(torch.isfinite(r["auc"]).all()) and 0 <= r["clean"]["auc"] <= 1


@pytest.mark.gpu
def test_rejections():
    from unidefense_b200 import ops
    from unidefense_b200.fourier import FourierHeatMap
    model = _model("r18")
    (x, lab), = _batches(sizes=(4,))
    for kw, match in ((dict(radius=0), "radius"), (dict(radius=1.5), "radius"), (dict(stride=0), "stride"),
                      (dict(eps=-1.0), "eps"), (dict(eps=float("nan")), "eps"), (dict(eps=float("inf")), "eps")):
        args = dict(eps=1.0)
        args.update(kw)
        with pytest.raises(ValueError, match=match):
            FourierHeatMap(model, **args)
    hm = FourierHeatMap(model, 1.0, radius=2)
    with pytest.raises(ValueError, match="eps"):
        hm.eps = -0.5
    assert hm.eps == 1.0
    with pytest.raises(RuntimeError, match="train mode"):
        FourierHeatMap(model.train(), 1.0, radius=2)([(x, lab)])
    model.eval()
    with pytest.raises(RuntimeError, match="CUDA fp32"):
        hm([(x.cpu(), lab)])
    with pytest.raises(RuntimeError, match="CUDA fp32"):
        hm([(x.double(), lab)])
    with pytest.raises(ValueError, match=r"\[N, C, H, W\]"):
        hm([(x[0], lab)])
    with pytest.raises(ValueError, match="labels for a batch"):
        hm([(x, lab[:2])])
    with pytest.raises(ValueError, match="every batch of a call"):
        hm([(x, lab), (x[..., :32, :32].contiguous(), lab)])
    for seed in (-1, 2 ** 64):
        with pytest.raises(ValueError, match="seed"):
            hm([(x, lab)], seed=seed)
    for ids in (torch.arange(3, device="cuda"), torch.arange(4, device="cuda", dtype=torch.int32), [0, 1, 2, 3]):
        with pytest.raises(ValueError, match="ids"):
            hm([(x, lab, ids)])
    with pytest.raises(ValueError, match="no batches"):
        hm([])
    with pytest.raises(ValueError, match="Nyquist"):
        FourierHeatMap(model, 1.0, radius=4, stride=9)([(x, lab)])
    with pytest.raises(ValueError, match="too small"):
        FourierHeatMap(model, 1.0, radius=40)([(x, lab)])
    y = torch.empty_like(x)
    f, e, s = _i32(0), torch.ones(1, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda")
    good = torch.zeros(1, 2, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="freqs"):
        ops.fourier_perturb(x, y, good.long(), f, e, None, s, LO, HI)
    with pytest.raises(ValueError, match="freqs"):
        ops.fourier_perturb(x, y, good[:, :1], f, e, None, s, LO, HI)
    with pytest.raises(ValueError, match="seed"):
        ops.fourier_perturb(x, y, good, f, e, None, s.int(), LO, HI)
    with pytest.raises(ValueError, match="one \\[N, C, H, W\\] shape"):
        ops.fourier_perturb(x, y[:2], good, f, e, None, s, LO, HI)
    with pytest.raises(RuntimeError, match="overlaps"):
        ops.fourier_perturb(x, x, good, f, e, None, s, LO, HI)
