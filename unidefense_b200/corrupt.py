"""Corruption-robustness evaluation of the UniDefense models: the image degradations of DeeperForensics-1.0 and
LipForensics (colour saturation, contrast, block-wise occlusion, Gaussian noise, Gaussian blur, pixelation, JPEG
compression) at five severities each, as CUDA kernels, and the accuracy / AUC table over a test set.

    from unidefense_b200 import corrupt
    y = corrupt.apply(x, "jpeg", severity=3)                      # JPEG at quality 50
    table = corrupt.evaluate(model.eval(), batches)                # {"clean": {"acc", "auc", "n"}, "jpeg": {1: ...}}

x is fp32 [N, 3, H, W], channels R, G, B, values in [lo, hi] (the reference's Normalize(0.5, 0.5) gives [-1, 1]).
Every corruption quantises to 8-bit levels, corrupts, and returns values on the 8-bit grid, as a decoded frame would
be; the exact definitions are in include/unidefense_b200.h (ud_corrupt).  Noise and block are random, keyed by a
per-sample int64 id and a uint64 seed rather than by batch position, so image i gets the same corruption in any batch
size and on any rank.  Video (H.264) compression is not offered: JPEG is the compression row.
"""
import torch

from . import ops
from ._evaluator import auc, check_call, p_fake, tally  # noqa: F401  (auc is part of this module's API)

_scores = p_fake        # this reader's earlier name here, which existing tests and scripts import

LEVELS = {
    "saturation": (0.4, 0.3, 0.2, 0.1, 0.0),     # chroma scale
    "contrast": (0.85, 0.725, 0.6, 0.475, 0.35),  # level scale
    "block": (16, 32, 48, 64, 80),                # 8x8 squares set to mid-grey
    "noise": (0.001, 0.002, 0.005, 0.01, 0.05),   # variance, in YCbCr / 255
    "blur": (7, 9, 13, 17, 21),                   # Gaussian kernel size, sigma = k/6
    "pixelate": (2, 3, 4, 5, 6),                  # cell size
    "jpeg": (90, 70, 50, 30, 10),                 # quality, 4:2:0
}
KINDS = tuple(LEVELS)


def _check_kind_severity(kind, severity):
    if kind not in LEVELS:
        raise ValueError(f"corrupt: kind must be one of {KINDS}, got {kind!r}")
    if isinstance(severity, bool) or not isinstance(severity, int) or not 1 <= severity <= 5:
        raise ValueError(f"corrupt: severity must be an int in 1..5, got {severity!r}")


def _check_rgb(x):
    if x.shape[1] != 3:
        raise ValueError(f"corrupt: x must be [N, 3, H, W] RGB, got {tuple(x.shape)}")


def apply(x, kind, severity, ids=None, seed=0, lo=-1.0, hi=1.0):
    """Corrupt a batch: `kind` from KINDS at `severity` 1..5 (LEVELS[kind][severity - 1]).  ids: int64 [N] per-sample
    keys of the random kinds (None: 0..N-1); seed: uint64.  Returns a new tensor; no gradient flows through it."""
    _check_kind_severity(kind, severity)
    x, _, _ = check_call("corrupt", None, x)
    _check_rgb(x)
    if ids is None:
        ids = torch.arange(x.shape[0], device=x.device)
    return ops.corrupt(x, kind, LEVELS[kind][severity - 1], ids, seed, lo, hi)


def evaluate(model, batches, kinds=KINDS, severities=(1, 2, 3, 4, 5), seed=0, lo=-1.0, hi=1.0):
    """Accuracy and AUC of a binary detector on clean and corrupted inputs.

    batches yields (x, labels) or (x, labels, ids): x CUDA fp32 [N, 3, H, W], labels {0 real, 1 fake}, ids int64 [N]
    (default: the running sample index over the iterable).  Per batch: one clean forward and one forward per
    (kind, severity), under no_grad and the caller's autocast.  The model must be in eval mode.  Returns
    {"clean": {"acc", "auc", "n"}, kind: {severity: {"acc", "auc", "n"}}}; the metrics are computed on the device and
    read once at the end."""
    kinds, severities = tuple(kinds), tuple(severities)
    for k in kinds:
        for s in severities:
            _check_kind_severity(k, s)
    keys = ["clean"] + [(k, s) for k in kinds for s in severities]

    def score(x, labels, ids, _):
        _check_rgb(x)
        ps, hits = [], []
        for key in keys:
            xin = x if key == "clean" else apply(x, key[0], key[1], ids, seed, lo, hi)
            p, pred = p_fake(model(xin)["cls_out"])
            ps.append(p)
            hits.append(pred == labels)
        return torch.stack(ps), torch.stack(hits)

    with torch.no_grad():
        stats, n = tally("corrupt.evaluate", model, batches, score)
    accs, aucs = stats.tolist()
    table = {}
    for key, acc, a in zip(keys, accs, aucs):
        row = {"acc": acc, "auc": a, "n": n}
        if key == "clean":
            table["clean"] = row
        else:
            table.setdefault(key[0], {})[key[1]] = row
    return table
