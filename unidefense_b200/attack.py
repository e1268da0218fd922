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

import torch
import torch.nn.functional as F

from . import ops
from ._evaluator import GraphedEvaluator, check_call, predicted


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


class PGD(GraphedEvaluator):
    """Projected gradient descent (ascent on the loss) with random restarts and best-iterate tracking.  The captured
    graphs live on this object (deleting it frees them); a new eps or alpha on a seen shape reuses them."""
    name = "PGD"

    def __init__(self, model, norm="linf", steps=10, restarts=1, random_start=True, lo=-1.0, hi=1.0):
        if norm not in ops.ATTACK_NORMS:
            raise ValueError(f"PGD: norm must be one of {sorted(ops.ATTACK_NORMS)}, got {norm!r}")
        if int(steps) < 1 or int(restarts) < 1:
            raise ValueError(f"PGD: steps ({steps}) and restarts ({restarts}) must be >= 1")
        super().__init__(model, lo, hi)
        self.norm = norm
        self.steps, self.restarts, self.random_start = int(steps), int(restarts), bool(random_start)

    # ---- the objective ------------------------------------------------------------------------------------------
    @staticmethod
    def _loss_and_miss(logits, labels):
        logits = logits.float()
        if logits.shape[1] == 1:
            loss = F.binary_cross_entropy_with_logits(logits[:, 0], labels.float(), reduction="none")
        else:
            loss = F.cross_entropy(logits, labels, reduction="none")
        return loss, predicted(logits) != labels

    def _score(self, st, logits, loss, miss):
        """Logits of the best iterate and the fooled flags; runs before ud_attack_step updates best_loss."""
        imp = loss > st.best_loss
        st.best_logits.copy_(torch.where(imp[:, None], logits.float(), st.best_logits))
        st.fooled.logical_or_(miss)

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

    def _best_logits(self, st):
        """A first forward finds the number of logits K of the best_logits buffer."""
        with self._autocast(st), torch.no_grad():
            K = self.model(st.x_adv)["cls_out"].shape[1]
        st.best_logits = torch.zeros(st.x0.shape[0], K, device=st.x0.device)

    # ---- capture --------------------------------------------------------------------------------------------------
    def _state(self, st, x, labels):
        N = x.shape[0]
        st.x0, st.x_adv, st.x_best = x.clone(), x.clone(), x.clone()
        st.labels = labels.clone()
        st.eps = torch.zeros(N, device=x.device)
        st.alpha = torch.zeros(N, device=x.device)
        st.best_loss = torch.full((N,), -math.inf, device=x.device)
        st.fooled = torch.zeros(N, dtype=torch.bool, device=x.device)
        st.step, st.final = self._capture(st, self._iteration, self._final, prepare=self._best_logits)

    # ---- the attack -------------------------------------------------------------------------------------------------
    def __call__(self, x, labels, eps=16 / 255, alpha=None):
        x, labels, key = check_call(self.name, self.model, x, labels)
        eps = float(eps)
        if not eps >= 0.0:
            raise ValueError(f"PGD: eps must be >= 0, got {eps}")
        alpha = 2.5 * eps / self.steps if alpha is None else float(alpha)
        st = self._graphed(key, x, labels)
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
