"""Batched PGD / FGSM robustness evaluation of the UniDefense models.

    atk = attack.PGD(model, norm="linf", steps=10, restarts=1, random_start=True, lo=-1.0, hi=1.0)
    res = atk(x, labels, eps=16/255)          # alpha default 2.5*eps/steps
    res["x_adv"], res["fooled"], res["best_loss"], res["logits"]

Untargeted: each sample ascends its own loss (cross-entropy, or BCE-with-logits when num_classes == 1) within the
eps-ball around x (L-inf or L2) and the input range [lo, hi].  The inputs follow the reference's Normalize(0.5, 0.5),
so [lo, hi] = [-1, 1] and eps is in input units (8/255 in pixels is 16/255 here).  FGSM is PGD(model, steps=1,
random_start=False) called with alpha=eps.

One iteration (forward at the current iterate, per-sample loss, d loss / dx, ud_attack_step: select + step + projection)
is captured as a CUDA graph once per input shape and autocast state and replayed `steps` times per restart; one more
captured forward plus a select-only step scores the final iterate.  Across restarts and iterates each sample keeps the
iterate of highest loss.  The caller's torch.autocast context applies (bf16 evaluation needs no option).
"""
import math
import types

import torch
import torch.nn.functional as F

from . import ops

_capture_streams = {}       # one side stream per device: warm-up and capture share it, and with it the op workspaces


def _capture_stream(device):
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _capture_streams:
        _capture_streams[idx] = torch.cuda.Stream(device=idx)
    return _capture_streams[idx]


def _random_start(x0, eps, norm, lo, hi):
    """Uniform in the L-inf ball, or a Gaussian direction at radius eps*U(0, 1) for L2 (oracle/attack.py)."""
    e = eps.view(-1, *([1] * (x0.dim() - 1)))
    if norm == "linf":
        r = torch.rand(x0.shape, dtype=x0.dtype, device=x0.device)
        return torch.clamp(x0 + (r * 2 - 1) * e, lo, hi)
    z = torch.randn(x0.shape, dtype=x0.dtype, device=x0.device)
    r = torch.rand(x0.shape[0], dtype=x0.dtype, device=x0.device)
    z = z / (z.flatten(1).norm(dim=1) + 1e-12).view_as(e)
    return torch.clamp(x0 + z * (eps * r).view_as(e), lo, hi)


class PGD:
    """Projected gradient descent (ascent on the loss) with random restarts and best-iterate tracking.  The captured
    graphs live on this object (deleting it frees them); a new eps or alpha on a seen shape reuses them."""

    def __init__(self, model, norm="linf", steps=10, restarts=1, random_start=True, lo=-1.0, hi=1.0):
        if norm not in ops.ATTACK_NORMS:
            raise ValueError(f"PGD: norm must be one of {sorted(ops.ATTACK_NORMS)}, got {norm!r}")
        if int(steps) < 1 or int(restarts) < 1:
            raise ValueError(f"PGD: steps ({steps}) and restarts ({restarts}) must be >= 1")
        if not float(lo) <= float(hi):
            raise ValueError(f"PGD: lo={lo} > hi={hi}")
        self.model, self.norm = model, norm
        self.steps, self.restarts, self.random_start = int(steps), int(restarts), bool(random_start)
        self.lo, self.hi = float(lo), float(hi)
        self._graphs = {}

    # ---- the objective ------------------------------------------------------------------------------------------
    @staticmethod
    def _loss_and_miss(logits, labels):
        logits = logits.float()
        if logits.shape[1] == 1:
            z = logits[:, 0]
            return F.binary_cross_entropy_with_logits(z, labels.float(), reduction="none"), (z > 0).long() != labels
        return F.cross_entropy(logits, labels, reduction="none"), logits.argmax(dim=1) != labels

    def _score(self, st, logits, loss, miss):
        """Logits of the best iterate and the fooled flags; runs before ud_attack_step updates best_loss."""
        imp = loss > st.best_loss
        st.best_logits.copy_(torch.where(imp[:, None], logits.float(), st.best_logits))
        st.fooled.logical_or_(miss)

    def _autocast(self, st):
        return torch.autocast("cuda", dtype=st.amp_dtype, enabled=st.amp_dtype is not None, cache_enabled=False)

    def _iteration(self, st):
        with self._autocast(st), torch.enable_grad():
            xin = st.x_adv.detach().requires_grad_()
            logits = self.model(xin)["cls_out"]
            loss, miss = self._loss_and_miss(logits, st.labels)
            g, = torch.autograd.grad(loss.sum(), xin)
        loss = loss.detach()
        self._score(st, logits.detach(), loss, miss)
        ops.attack_step(st.x0, st.x_adv, g.contiguous(), loss, st.best_loss, st.x_best, st.eps, st.alpha, self.lo,
                        self.hi, self.norm)

    def _final(self, st):
        with self._autocast(st), torch.no_grad():
            logits = self.model(st.x_adv)["cls_out"]
            loss, miss = self._loss_and_miss(logits, st.labels)
        self._score(st, logits, loss, miss)
        ops.attack_step(st.x0, st.x_adv, None, loss, st.best_loss, st.x_best, None, None, self.lo, self.hi, self.norm)

    # ---- capture --------------------------------------------------------------------------------------------------
    def _capture(self, x, labels, amp_dtype):
        N = x.shape[0]
        st = types.SimpleNamespace(amp_dtype=amp_dtype)
        st.x0, st.x_adv, st.x_best = x.clone(), x.clone(), x.clone()
        st.labels = labels.clone()
        st.eps = torch.zeros(N, device=x.device)
        st.alpha = torch.zeros(N, device=x.device)
        st.best_loss = torch.full((N,), -math.inf, device=x.device)
        st.fooled = torch.zeros(N, dtype=torch.bool, device=x.device)
        side = _capture_stream(x.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            # warm-up: first calls build FFT tables with a synchronous copy and grow the op workspaces (header
            # conventions); none of that may happen inside the capture
            with self._autocast(st), torch.no_grad():
                K = self.model(st.x_adv)["cls_out"].shape[1]
            st.best_logits = torch.zeros(N, K, device=x.device)
            for _ in range(2):
                self._iteration(st)
                self._final(st)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        st.step = torch.cuda.CUDAGraph()
        with torch.cuda.graph(st.step, stream=side, capture_error_mode="thread_local"):
            self._iteration(st)
        st.final = torch.cuda.CUDAGraph()
        with torch.cuda.graph(st.final, pool=st.step.pool(), stream=side, capture_error_mode="thread_local"):
            self._final(st)
        return st

    # ---- the attack -------------------------------------------------------------------------------------------------
    def __call__(self, x, labels, eps=16 / 255, alpha=None):
        if any(m.training for m in self.model.modules()):
            raise RuntimeError("PGD: the model is in train mode; call model.eval() first (every replay would move the "
                               "BatchNorm running statistics and draw dropout)")
        if not torch.is_tensor(x) or not x.is_cuda or x.dtype != torch.float32:
            raise RuntimeError("PGD: x must be a CUDA fp32 tensor")
        if x.device.index != torch.cuda.current_device():
            raise RuntimeError(f"PGD: x is on cuda:{x.device.index} but the current device is "
                               f"cuda:{torch.cuda.current_device()}")
        eps = float(eps)
        if not eps >= 0.0:
            raise ValueError(f"PGD: eps must be >= 0, got {eps}")
        alpha = 2.5 * eps / self.steps if alpha is None else float(alpha)
        labels = torch.as_tensor(labels).to(device=x.device, dtype=torch.long).reshape(-1)
        if x.dim() < 2 or labels.numel() != x.shape[0]:
            raise ValueError(f"PGD: {labels.numel()} labels for a batch of {x.shape[0] if x.dim() else 0}")
        x = x.detach().contiguous()
        amp = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else None
        key = (tuple(x.shape), amp, x.device.index)
        st = self._graphs.get(key)
        if st is None:
            st = self._graphs[key] = self._capture(x, labels, amp)
        st.x0.copy_(x)
        st.x_best.copy_(x)
        st.labels.copy_(labels)
        st.eps.fill_(eps)
        st.alpha.fill_(alpha)
        st.best_loss.fill_(-math.inf)
        st.best_logits.fill_(math.nan)
        st.fooled.zero_()
        for _ in range(self.restarts):
            st.x_adv.copy_(_random_start(st.x0, st.eps, self.norm, self.lo, self.hi) if self.random_start else st.x0)
            for _ in range(self.steps):
                st.step.replay()
            st.final.replay()
        return {"x_adv": st.x_best.clone(), "fooled": st.fooled.clone(), "best_loss": st.best_loss.clone(),
                "logits": st.best_logits.clone()}
