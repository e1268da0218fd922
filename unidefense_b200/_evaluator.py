"""What the evaluators (attack.PGD, corrupt.evaluate, explain.*, fourier.FourierHeatMap) share: the call checks, the
readers of a detector's head, the captured-graph cache and the tally of a batch stream.

An evaluator that replays graphs (GraphedEvaluator) captures two of them per input shape, autocast state and device,
and keeps them in self._graphs under the key (shape, autocast dtype or None, device index).  Warm-up and capture run
on one side stream per device: the first calls build FFT tables with a synchronous copy and grow the op workspaces,
which are per stream (_lib.workspace); none of that may happen inside a capture.  The two graphs share one pool.
"""
import types

import torch
import torch.nn.functional as F

from ._lib import require_ids

_side_streams = {}


def check_call(name, model, x, labels=None):
    """Check that the model (unless None) is in eval mode, x is a CUDA fp32 [N, C, H, W] tensor on the current device
    and labels (unless None) hold N classes.  -> (x detached and contiguous, labels as int64 [N] or None, the graph
    key).  `name` starts every message."""
    if model is not None and any(m.training for m in model.modules()):
        raise RuntimeError(f"{name}: the model is in train mode; call model.eval() first (BatchNorm would use and move "
                           "batch statistics, and dropout would draw)")
    if not torch.is_tensor(x) or not x.is_cuda or x.dtype != torch.float32:
        raise RuntimeError(f"{name}: x must be a CUDA fp32 tensor")
    if x.device.index != torch.cuda.current_device():
        raise RuntimeError(f"{name}: x is on cuda:{x.device.index} but the current device is "
                           f"cuda:{torch.cuda.current_device()}")
    if x.dim() != 4:
        raise ValueError(f"{name}: x must be [N, C, H, W], got {tuple(x.shape)}")
    if labels is not None:
        labels = torch.as_tensor(labels).to(device=x.device, dtype=torch.long).reshape(-1)
        if labels.numel() != x.shape[0]:
            raise ValueError(f"{name}: {labels.numel()} labels for a batch of {x.shape[0]}")
    amp = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else None
    return x.detach().contiguous(), labels, (tuple(x.shape), amp, x.device.index)


def predicted(logits):
    """The predicted class: logit > 0 for one logit, else the argmax."""
    logits = logits.float()
    return (logits[:, 0] > 0).long() if logits.shape[1] == 1 else logits.argmax(dim=1)


def p_fake(logits):
    """P(fake) and the predicted class of a binary detector: sigmoid of one logit, or softmax column 1 of two."""
    logits = logits.float()
    if logits.shape[1] == 1:
        return torch.sigmoid(logits[:, 0]), predicted(logits)
    if logits.shape[1] == 2:
        return torch.softmax(logits, dim=1)[:, 1], predicted(logits)
    raise ValueError(f"a binary detector has 1 or 2 logits, got {logits.shape[1]}")


def log_p(logits, target):
    """F = log p(target | logits) per sample, in fp32: logsigmoid(+-z) of one logit, else log_softmax."""
    logits = logits.float()
    if logits.shape[1] == 1:
        z = logits[:, 0]
        return F.logsigmoid(torch.where(target == 1, z, -z))
    return torch.log_softmax(logits, dim=1).gather(1, target[:, None])[:, 0]


class GraphedEvaluator:
    """Owns the captured graphs of an evaluator (deleting it frees them).  A subclass sets `name`, the start of its
    messages, and `_state(st, x, ...)`, which fills the state of one key and captures its graphs."""

    def __init__(self, model, lo, hi):
        if not float(lo) <= float(hi):
            raise ValueError(f"{self.name}: lo={lo} > hi={hi}")
        self.model, self.lo, self.hi = model, float(lo), float(hi)
        self._graphs = {}

    def _graphed(self, key, x, *args):
        st = self._graphs.get(key)
        if st is None:
            st = types.SimpleNamespace(amp_dtype=key[1])
            self._state(st, x, *args)
            self._graphs[key] = st
        return st

    @staticmethod
    def _autocast(st):
        return torch.autocast("cuda", dtype=st.amp_dtype, enabled=st.amp_dtype is not None, cache_enabled=False)

    @staticmethod
    def _capture(st, first, second, prepare=None):
        """-> the graphs of first(st) and second(st), in one pool.  Warm-up, on the side stream: prepare(st), then
        first and second twice."""
        idx = torch.cuda.current_device()           # x's device (check_call)
        if idx not in _side_streams:
            _side_streams[idx] = torch.cuda.Stream(device=idx)
        side = _side_streams[idx]
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            if prepare is not None:
                prepare(st)
            for _ in range(2):
                first(st)
                second(st)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g1 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g1, stream=side, capture_error_mode="thread_local"):
            first(st)
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2, pool=g1.pool(), stream=side, capture_error_mode="thread_local"):
            second(st)
        return g1, g2


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


def tally(name, model, batches, score):
    """Accuracy and AUC of R rows of scores over batches of (x, labels) or (x, labels, ids), ids defaulting to the
    running sample index: score(x, labels, ids, key) of each batch, checked by check_call, returns its p(fake) and hits
    [R, N].  -> (fp64 [2, R]: the rows' acc and auc, read to the host once; the sample count n)."""
    p, hits, all_labels, n = [], [], [], 0
    for batch in batches:
        x, labels, key = check_call(name, model, batch[0], batch[1])
        if labels is None:
            raise ValueError(f"{name}: every batch needs labels")
        ids = require_ids(batch[2] if len(batch) > 2 else None, x, name)
        if ids is None:
            ids = torch.arange(n, n + x.shape[0], device=x.device)
        pb, hb = score(x, labels, ids, key)
        p.append(pb)
        hits.append(hb)
        all_labels.append(labels)
        n += x.shape[0]
    if n == 0:
        raise ValueError(f"{name}: no batches")
    stats = torch.stack([torch.cat(hits, -1).double().mean(-1), auc(torch.cat(p, -1), torch.cat(all_labels))])
    return stats.cpu(), n
