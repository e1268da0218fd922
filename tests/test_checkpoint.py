"""Checkpoint interchange with the reference engines (SURVEY.md §8f row 4): unidefense_b200.checkpoint.

CPU tests.  The cross-load cases check against the reference classes' state_dict layout recorded in
tests/golden/full_<arch>.pt."""
import io
import os

import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

CTOR = {"r18": ("UDR18", dict(num_classes=2, drop_rate=0.5)),
        "r50": ("UDR50", dict(extractor="resnet50", num_classes=2, drop_rate=0.5)),
        "eb4": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2, drop_rate=0.2))}


def _ours(arch):
    from unidefense_b200.model import load_model
    name, kw = CTOR[arch]
    return load_model(name)(**kw)


def _randomise(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for v in model.state_dict().values():
            if v.dtype.is_floating_point:
                v.copy_(torch.randn(v.shape, generator=g))
            else:
                v.fill_(seed)


@pytest.mark.parametrize("arch", ["r18", "eb4"])
def test_self_round_trip_and_layout(arch):
    from unidefense_b200 import checkpoint as CK
    a = _ours(arch)
    _randomise(a, 3)
    buf = io.BytesIO()
    CK.save_reference_checkpoint(a, buf, step=7, best_step=5, best_auc=0.91, best_acc=0.88)
    buf.seek(0)
    raw = torch.load(buf, map_location="cpu", weights_only=True)
    assert list(raw) == ["step", "best_step", "best_auc", "best_acc", "model"]          # forgery_engine.py:217-223
    assert all(v.is_contiguous() for v in raw["model"].values())                         # also the channels-last 3x3 weight
    assert list(raw["model"]) == list(a.state_dict())
    b = _ours(arch)
    buf.seek(0)
    meta = CK.load_reference_checkpoint(b, buf)
    assert meta == dict(step=7, best_step=5, best_auc=0.91, best_acc=0.88)
    for (k, u), (k2, v) in zip(a.state_dict().items(), b.state_dict().items()):
        assert k == k2 and torch.equal(u, v), k
    buf.seek(0)
    assert CK.verify(b, buf)[1] == len(a.state_dict())


def test_ddp_prefix_bare_state_dict_and_errors():
    from unidefense_b200 import checkpoint as CK
    a, b = _ours("r18"), _ours("r18")
    _randomise(a, 1)
    buf = io.BytesIO()
    torch.save({"module." + k: v for k, v in a.state_dict().items()}, buf)              # bare + DDP-prefixed
    buf.seek(0)
    assert CK.load_reference_checkpoint(b, buf) == {}
    assert all(torch.equal(u, v) for u, v in zip(a.state_dict().values(), b.state_dict().values()))
    sd = dict(a.state_dict())
    sd.pop("fuse_coef")
    sd["classifier.fc.weight"] = torch.zeros(3, 512)
    sd["not_a_key"] = torch.zeros(1)
    buf = io.BytesIO()
    torch.save({"model": sd, "best_step": 1}, buf)
    buf.seek(0)
    with pytest.raises(RuntimeError) as e:
        CK.load_reference_checkpoint(b, buf)
    msg = str(e.value)
    assert "missing in file: fuse_coef" in msg and "unexpected in file: not_a_key" in msg and "classifier.fc.weight" in msg
    with pytest.raises(ValueError):
        buf = io.BytesIO()
        torch.save({"weights": 3}, buf)
        buf.seek(0)
        CK.load_reference_checkpoint(b, buf)


def _reference_state_dict(arch, seed):
    """A state_dict laid out as the reference class's: the key order and shapes make_golden.py recorded from it
    (tests/golden/full_<arch>.pt), BatchNorm counters int64 as torch keeps them, seeded values."""
    shapes = torch.load(os.path.join(GOLDEN, f"full_{arch}.pt"), weights_only=False)["state_dict_shapes"]
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, shape in shapes.items():
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.full(shape, seed, dtype=torch.int64)
        else:
            sd[k] = torch.randn(shape, generator=g)
    return sd


@pytest.mark.parametrize("arch", ["r18", "r50", "eb4"])
def test_cross_load_with_the_reference_layout(arch, tmp_path):
    """A file written the way the reference engine writes it loads strictly into the drop-in, and a file written by
    the drop-in passes the reference's strict load (forgery_engine.py:200-209: same keys, same shapes), keys in the
    reference order, tensors bit-identical."""
    from unidefense_b200 import checkpoint as CK
    ref_sd = _reference_state_dict(arch, 5)
    path = os.path.join(tmp_path, "best_model.bin")
    torch.save({"step": 12, "best_step": 10, "best_auc": 0.97, "best_acc": 0.93, "model": ref_sd}, path)
    ours = _ours(arch)
    meta = CK.load_reference_checkpoint(ours, path)
    assert meta["best_step"] == 10
    assert list(ours.state_dict()) == list(ref_sd)
    for (k, u), (k2, v) in zip(ref_sd.items(), ours.state_dict().items()):
        assert k == k2 and u.shape == v.shape and u.dtype == v.dtype and torch.equal(u, v), k
    assert CK.verify(ours, path)[1] == len(ref_sd)
    # and back: the drop-in's file against the reference's strict load_state_dict
    _randomise(ours, 9)
    back = os.path.join(tmp_path, "latest_model.bin")
    CK.save_reference_checkpoint(ours, back, step=13, best_step=10, best_auc=0.97, best_acc=0.93)
    ckpt = torch.load(back, map_location="cpu")
    assert list(ckpt["model"]) == list(ref_sd)
    for (k, u), v in zip(ckpt["model"].items(), ours.state_dict().values()):
        assert u.shape == ref_sd[k].shape and u.dtype == ref_sd[k].dtype and torch.equal(u, v), k
    assert round(ckpt.get("best_auc", -1), 4) == 0.97                                   # the engine's print statement
