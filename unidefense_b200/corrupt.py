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


def _check_input(x):
    if not torch.is_tensor(x) or not x.is_cuda:
        raise RuntimeError("corrupt: x must be a CUDA tensor (no CPU fallback)")
    if x.dtype != torch.float32:
        raise RuntimeError(f"corrupt: x must be fp32, got {x.dtype}")
    if x.dim() != 4 or x.shape[1] != 3:
        raise ValueError(f"corrupt: x must be [N, 3, H, W] RGB, got {tuple(x.shape)}")
    if x.device.index != torch.cuda.current_device():
        raise RuntimeError(f"corrupt: x is on cuda:{x.device.index} but the current device is "
                           f"cuda:{torch.cuda.current_device()}")


def apply(x, kind, severity, ids=None, seed=0, lo=-1.0, hi=1.0):
    """Corrupt a batch: `kind` from KINDS at `severity` 1..5 (LEVELS[kind][severity - 1]).  ids: int64 [N] per-sample
    keys of the random kinds (None: 0..N-1); seed: uint64.  Returns a new tensor; no gradient flows through it."""
    _check_kind_severity(kind, severity)
    _check_input(x)
    if ids is None:
        ids = torch.arange(x.shape[0], device=x.device)
    return ops.corrupt(x.contiguous(), kind, LEVELS[kind][severity - 1], ids, seed, lo, hi)


def _scores(logits):
    """P(fake) and the predicted label from [N, 2] logits (softmax column 1, argmax) or [N, 1] (sigmoid, logit > 0)."""
    logits = logits.float()
    if logits.shape[1] == 1:
        return torch.sigmoid(logits[:, 0]), (logits[:, 0] > 0).long()
    if logits.shape[1] == 2:
        return torch.softmax(logits, dim=1)[:, 1], logits.argmax(dim=1)
    raise ValueError(f"corrupt.evaluate: a binary detector has 1 or 2 logits, got {logits.shape[1]}")


def auc(scores, labels):
    """Mann-Whitney AUC with tie-averaged ranks, on the device and without a host synchronisation (NaN when one class
    is absent).  Label 1 is the positive (fake) class.  scores [..., n] against labels [n]: one AUC per row of the
    last dimension.  Every partial sum is a multiple of 1/2 below 2^53, so a row scores the same alone or batched."""
    n = scores.shape[-1]
    v, order = torch.sort(scores.double(), dim=-1)
    pos = (labels[order] == 1).double()
    idx = torch.arange(n, device=scores.device)
    new = torch.ones(v.shape, dtype=torch.bool, device=scores.device)
    new[..., 1:] = v[..., 1:] != v[..., :-1]
    end = torch.ones_like(new)
    end[..., :-1] = new[..., 1:]
    first = torch.cummax(torch.where(new, idx, 0), -1).values
    last = torch.flip(torch.cummin(torch.flip(torch.where(end, idx, n - 1), [-1]), -1).values, [-1])
    rank = (first + last).double() / 2 + 1
    n_pos = pos.sum(-1)
    n_neg = n - n_pos
    return ((rank * pos).sum(-1) - n_pos * (n_pos + 1) / 2) / (n_pos * n_neg)


def evaluate(model, batches, kinds=KINDS, severities=(1, 2, 3, 4, 5), seed=0, lo=-1.0, hi=1.0):
    """Accuracy and AUC of a binary detector on clean and corrupted inputs.

    batches yields (x, labels) or (x, labels, ids): x CUDA fp32 [N, 3, H, W], labels {0 real, 1 fake}, ids int64 [N]
    (default: the running sample index over the iterable).  Per batch: one clean forward and one forward per
    (kind, severity), under no_grad and the caller's autocast.  The model must be in eval mode.  Returns
    {"clean": {"acc", "auc", "n"}, kind: {severity: {"acc", "auc", "n"}}}; the metrics are computed on the device and
    read once at the end."""
    if any(m.training for m in model.modules()):
        raise RuntimeError("corrupt.evaluate: the model is in train mode; call model.eval() first (BatchNorm would use "
                           "batch statistics and dropout would draw)")
    kinds, severities = tuple(kinds), tuple(severities)
    for k in kinds:
        for s in severities:
            _check_kind_severity(k, s)
    keys = ["clean"] + [(k, s) for k in kinds for s in severities]
    scores = {key: [] for key in keys}
    hits = {key: [] for key in keys}
    all_labels = []
    n = 0
    with torch.no_grad():
        for batch in batches:
            x, labels = batch[0], batch[1]
            ids = batch[2] if len(batch) > 2 else None
            _check_input(x)
            N = x.shape[0]
            labels = labels.to(x.device).long()
            if ids is None:
                ids = torch.arange(n, n + N, device=x.device)
            n += N
            all_labels.append(labels)
            for key in keys:
                xin = x if key == "clean" else apply(x, key[0], key[1], ids, seed, lo, hi)
                p, pred = _scores(model(xin)["cls_out"])
                scores[key].append(p)
                hits[key].append(pred == labels)
    if n == 0:
        raise ValueError("corrupt.evaluate: no batches")
    labels = torch.cat(all_labels)
    stats = torch.stack([torch.stack([torch.cat(hits[k]).double().mean(), auc(torch.cat(scores[k]), labels)])
                         for k in keys]).tolist()
    table = {}
    for key, (acc, a) in zip(keys, stats):
        row = {"acc": acc, "auc": a, "n": n}
        if key == "clean":
            table["clean"] = row
        else:
            table.setdefault(key[0], {})[key[1]] = row
    return table
