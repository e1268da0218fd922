"""Image corruptions: ud_corrupt against oracle/corrupt.py for every kind x severity at 64², 299² and 380² with
N in {1, 4, 32} (saturation, contrast, block and pixelate bit-identical; noise, blur and jpeg equal on every certain
element and within one level on the uncertain ones), reproducibility, per-sample keying, unaligned views, and
corrupt.evaluate against an eager loop of apply + forward with the AUC of scipy's rank formula."""
import functools

import numpy as np
import pytest
import torch

import procedural as P
from oracle import corrupt as C

LO, HI = -1.0, 1.0
EXACT = ("saturation", "contrast", "block", "pixelate")
SEED = 0x123456789ABCDEF0


@functools.lru_cache(maxsize=None)
def _images(H, W, N=32):
    return C.test_images(N, H, W, seed=0)


@functools.lru_cache(maxsize=4)
def _oracle(kind, sev, H, W):
    return C.corrupt(_images(H, W), kind, C.LEVELS[kind][sev - 1], ids=np.arange(32), seed=SEED)


def _levels(y):
    return C.to_levels(np.asarray(y), LO, HI).astype(np.int64)


def _compare(got, want, unc, what):
    got = got.cpu().numpy()
    if unc is None:
        assert np.array_equal(got, want), (what, int((got != want).sum()))
        return
    d = np.abs(_levels(got) - _levels(want))
    assert (d[~unc] == 0).all(), (what, int((d[~unc] != 0).sum()), np.argwhere((d != 0) & ~unc)[:5])
    assert d[unc].max(initial=0) <= 1, (what, int(d[unc].max()))
    assert unc.mean() <= 0.005, (what, unc.mean())


@pytest.mark.gpu
@pytest.mark.parametrize("size", [64, 299, 380])
@pytest.mark.parametrize("sev", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("kind", C.KINDS)
def test_kernel_matches_oracle(kind, sev, size):
    from unidefense_b200 import corrupt
    y_want, unc = _oracle(kind, sev, size, size)
    x = torch.from_numpy(_images(size, size)).cuda()
    for N in (1, 4, 32):
        y = corrupt.apply(x[:N], kind, sev, seed=SEED)
        assert y.shape == x[:N].shape and y.dtype == torch.float32 and not y.requires_grad
        _compare(y, y_want[:N], None if unc is None else unc[:N], (kind, sev, size, N))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", C.KINDS)
def test_odd_non_square_size(kind):
    from unidefense_b200 import corrupt
    xn = C.test_images(3, 45, 67, seed=8)
    x = torch.from_numpy(xn).cuda()
    for sev in (1, 5):
        want, unc = C.corrupt(xn, kind, C.LEVELS[kind][sev - 1], seed=3)
        _compare(corrupt.apply(x, kind, sev, seed=3), want, unc, (kind, sev))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", C.KINDS)
def test_reproducible_keyed_per_sample_and_unaligned(kind):
    from unidefense_b200 import corrupt
    x = torch.from_numpy(_images(299, 299)[:4]).cuda()
    ids = torch.tensor([7, 3, 10 ** 12, -5], device="cuda")
    y = corrupt.apply(x, kind, 3, ids=ids, seed=SEED)
    assert torch.equal(y, corrupt.apply(x, kind, 3, ids=ids, seed=SEED))
    for i in range(4):
        assert torch.equal(corrupt.apply(x[i:i + 1].clone(), kind, 3, ids=ids[i:i + 1], seed=SEED), y[i:i + 1])
    buf = torch.empty(x.numel() + 1, device="cuda")
    xu = buf[1:].view_as(x)                       # 4 bytes past a 16-byte boundary: the scalar paths
    xu.copy_(x)
    assert xu.data_ptr() % 16 == 4
    assert torch.equal(corrupt.apply(xu, kind, 3, ids=ids, seed=SEED), y)
    other = corrupt.apply(x, kind, 3, ids=ids, seed=SEED + 1)
    assert torch.equal(other, y) == (kind not in ("noise", "block"))
    x64 = torch.from_numpy(_images(64, 64)[:2]).cuda()
    assert torch.equal(corrupt.apply(x64, kind, 2), corrupt.apply(x64, kind, 2, ids=torch.arange(2, device="cuda")))


@pytest.mark.gpu
def test_apply_rejects_bad_inputs():
    from unidefense_b200 import corrupt
    x = torch.zeros(2, 3, 16, 16, device="cuda")
    with pytest.raises(RuntimeError, match="CUDA"):
        corrupt.apply(x.cpu(), "jpeg", 1)
    with pytest.raises(RuntimeError, match="fp32"):
        corrupt.apply(x.double(), "jpeg", 1)
    with pytest.raises(ValueError, match="RGB"):
        corrupt.apply(x[:, :2], "jpeg", 1)
    for sev in (0, 6, 2.0, True):
        with pytest.raises(ValueError, match="severity"):
            corrupt.apply(x, "jpeg", sev)
    with pytest.raises(ValueError, match="kind"):
        corrupt.apply(x, "h264", 1)
    with pytest.raises(RuntimeError, match="needs H, W > 10"):
        corrupt.apply(x[..., :10, :10], "blur", 5)


CTOR = {"eb4": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2, drop_rate=0.0, drop_connect_rate=0.0)),
        "r18": ("UDR18", dict(num_classes=2, drop_rate=0.0)),
        "eb4_bce": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=1, drop_rate=0.0, drop_connect_rate=0.0))}


def _model(arch):
    from unidefense_b200.model import load_model
    name, kw = CTOR[arch]
    model = load_model(name)(**kw)
    P.fill_state_dict_(model, salt=5)
    return model.cuda().eval()


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["r18", "eb4", "eb4_bce"])
def test_evaluate_matches_an_eager_loop(arch):
    from scipy.stats import rankdata
    from unidefense_b200 import corrupt
    model = _model(arch)
    R = 64
    xs = torch.from_numpy(_images(R, R, 12)).cuda()
    labels = torch.tensor([0, 1] * 6, device="cuda")
    batches = [(xs[:5], labels[:5]), (xs[5:], labels[5:])]
    kinds, sevs = ("jpeg", "noise", "block"), (1, 5)
    table = corrupt.evaluate(model, batches, kinds=kinds, severities=sevs, seed=4)
    y = labels.cpu().numpy()

    def metrics(logits):
        logits = logits.float().cpu()
        if logits.shape[1] == 1:
            s, pred = torch.sigmoid(logits[:, 0]), (logits[:, 0] > 0).long()
        else:
            s, pred = torch.softmax(logits, 1)[:, 1], logits.argmax(1)
        r = rankdata(s.double().numpy())
        npos = int(y.sum())
        a = (r[y == 1].sum() - npos * (npos + 1) / 2) / (npos * (len(y) - npos))
        return float((pred.numpy() == y).mean()), a

    with torch.no_grad():
        acc, a = metrics(torch.cat([model(b[0])["cls_out"] for b in batches]))
        assert table["clean"] == {"acc": acc, "auc": pytest.approx(a, abs=1e-12), "n": 12}
        for k in kinds:
            for s in sevs:
                logits = torch.cat([model(corrupt.apply(xs[i:j], k, s, ids=torch.arange(i, j, device="cuda"),
                                                        seed=4))["cls_out"] for i, j in ((0, 5), (5, 12))])
                acc, a = metrics(logits)
                assert table[k][s] == {"acc": acc, "auc": pytest.approx(a, abs=1e-12), "n": 12}, (k, s)
    # explicit ids equal the running index
    t2 = corrupt.evaluate(model, [(xs, labels, torch.arange(12, device="cuda"))], kinds=kinds, severities=sevs, seed=4)
    assert t2["noise"][5]["acc"] == table["noise"][5]["acc"]


@pytest.mark.gpu
def test_evaluate_under_bf16_autocast_runs():
    from unidefense_b200 import corrupt
    model = _model("r18")
    xs = torch.from_numpy(_images(64, 64, 4)).cuda()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        t = corrupt.evaluate(model, [(xs, torch.tensor([0, 1, 0, 1], device="cuda"))], kinds=("blur",), severities=(3,))
    assert set(t) == {"clean", "blur"} and 0 <= t["blur"][3]["auc"] <= 1


@pytest.mark.gpu
def test_evaluate_rejects_bad_inputs():
    from unidefense_b200 import corrupt
    model = _model("r18")
    xs = torch.from_numpy(_images(64, 64, 2)).cuda()
    lab = torch.tensor([0, 1], device="cuda")
    with pytest.raises(RuntimeError, match="train mode"):
        corrupt.evaluate(model.train(), [(xs, lab)])
    model.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        corrupt.evaluate(model, [(xs.cpu(), lab.cpu())])
    with pytest.raises(ValueError, match="severity"):
        corrupt.evaluate(model, [(xs, lab)], severities=(0,))
    with pytest.raises(ValueError, match="kind"):
        corrupt.evaluate(model, [(xs, lab)], kinds=("h264",))
