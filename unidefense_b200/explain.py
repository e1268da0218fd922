"""Attribution maps (Integrated Gradients, SmoothGrad) of the UniDefense models and their deletion / insertion
faithfulness scores.

    ig = explain.IntegratedGradients(model.eval(), steps=32, lo=-1.0, hi=1.0)
    r = ig(x, labels=None, baseline=None)         # {"attr", "map", "target", "f_x", "f_baseline", "delta"}
    sg = explain.SmoothGrad(model.eval(), draws=16, noise=0.15, lo=-1.0, hi=1.0)
    r = sg(x, labels=None, ids=None, seed=0)      # {"attr", "map", "target"}
    fa = explain.Faithfulness(model.eval(), points=16, lo=-1.0, hi=1.0)
    c = fa(x, r["map"], labels=None, baseline=None)   # {"deletion", "insertion": [N, K+1], "deletion_auc", "insertion_auc"}

The objective is F(x) = log p(target | x) (log_softmax of the two logits, or logsigmoid(+-z) of one), so one-logit and
two-logit heads mean the same thing; the target is `labels` when given, else the class predicted at x.  Both methods
accumulate sum_k w_k * grad F(p_k) over the path points p_k = b + alpha_k*(x - b) + sigma*eps_k:
 - Integrated Gradients: alpha_k = k/m (k = 0..m), trapezoid weights, attr = (x - b) * acc.  The baseline b is `lo`
   (the black image) by default, a float, or a tensor of x's shape (a blurred x, say).  delta = sum(attr) -
   (F(x) - F(b)) per sample is the completeness error; it falls as `steps` grows.
 - SmoothGrad: alpha_k = 1, sigma = noise*(hi - lo), w_k = 1/draws, attr = acc, no clamp (Smilkov et al.).  The noise
   is keyed by a per-sample int64 id and a uint64 seed (Philox4x32-10), so sample i gets the same noise at any batch
   size and on any rank.  SmoothGrad(draws=1, noise=0) is the vanilla gradient.
map = sum_c |attr_c|, [N, H, W].  Faithfulness ranks the pixels of any [N, H, W] map (descending, ties by pixel index,
NaN last); point j = 0..K of the deletion curve replaces the first floor(j*H*W/K) pixels (all channels) with the
baseline, the insertion curve starts from the baseline and restores them; the score is p(target | input) and the AUC
the trapezoid over j/K (after Petsiuk et al., RISE).  Exact definitions: include/unidefense_b200.h (ud_attrib_step).

One iteration (forward, F, d F / dx, ud_attrib_step) is captured as a CUDA graph once per input shape, autocast state
and device and replayed (_evaluator.GraphedEvaluator); so is one faithfulness point (the two masked inputs, their
no_grad forwards, the scores).  Nothing in a call synchronises with the host.  The caller's torch.autocast context
applies.
"""
import torch

from . import _lib as L
from . import ops
from ._evaluator import GraphedEvaluator, check_call, log_p as objective, predicted     # noqa: F401  (public)


class _Explainer(GraphedEvaluator):
    name = "explain"

    def _baseline(self, st, baseline, x):
        """Fill st.b from None (lo), a float or a tensor of x's shape on x's device."""
        if baseline is None:
            st.b.fill_(self.lo)
        elif torch.is_tensor(baseline):
            if baseline.shape != x.shape or baseline.dtype != torch.float32 or baseline.device != x.device:
                raise ValueError(f"{self.name}: baseline must be an fp32 tensor of x's shape {tuple(x.shape)} on "
                                 f"{x.device}, got {baseline.dtype} {tuple(baseline.shape)} on {baseline.device}")
            st.b.copy_(baseline)
        else:
            st.b.fill_(float(baseline))

    def _new_state(self, st, x):
        N = x.shape[0]
        st.x = x.clone()
        st.labels = torch.zeros(N, dtype=torch.long, device=x.device)
        st.use_labels = torch.zeros((), dtype=torch.bool, device=x.device)
        st.target = torch.zeros(N, dtype=torch.long, device=x.device)
        st.f_x = torch.zeros(N, device=x.device)

    def _target(self, st):
        """Forward at x: the target (the label, or the class predicted at x) and F(x)."""
        with self._autocast(st), torch.no_grad():
            logits = self.model(st.x)["cls_out"]
        st.target.copy_(torch.where(st.use_labels, st.labels, predicted(logits)))
        st.f_x.copy_(objective(logits, st.target))

    def _set_labels(self, st, labels):
        if labels is None:
            st.use_labels.fill_(False)
        else:
            st.labels.copy_(labels)
            st.use_labels.fill_(True)


class _Attribution(_Explainer):
    method = None

    def _tables(self):
        """-> (alpha, w) as float64 lists of the S path points."""
        raise NotImplementedError

    def _prologue(self, st):
        self._target(st)
        st.k.zero_()
        ops.attrib_step(st.x, st.bv, None, st.acc, st.p, st.attr, st.map, st.k, st.alpha, st.w, self.method,
                        st.sigma, st.ids, st.seed)

    def _iteration(self, st):
        with self._autocast(st), torch.enable_grad():
            xin = st.p.detach().requires_grad_()
            f = objective(self.model(xin)["cls_out"], st.target)
            g, = torch.autograd.grad(f.sum(), xin)
        if self.method == "ig":
            st.f_b.copy_(torch.where(st.k == 0, f.detach(), st.f_b))       # F at p_0 = b
        ops.attrib_step(st.x, st.bv, g.contiguous(), st.acc, st.p, st.attr, st.map, st.k, st.alpha, st.w, self.method,
                        st.sigma, st.ids, st.seed)
        st.k.add_(1)

    def _state(self, st, x):
        self._new_state(st, x)
        N, C, H, W = x.shape
        dev = x.device
        alpha, w = self._tables()
        st.alpha = torch.tensor(alpha, dtype=torch.float32, device=dev)
        st.w = torch.tensor(w, dtype=torch.float32, device=dev)
        st.k = torch.zeros(1, dtype=torch.int32, device=dev)
        st.acc, st.p, st.attr = (torch.zeros_like(x) for _ in range(3))
        st.map = torch.zeros(N, H, W, device=dev)
        st.f_b = torch.zeros(N, device=dev)
        st.b = torch.full_like(x, self.lo) if self.method == "ig" else None
        st.bv = st.b if self.method == "ig" else 0.0
        st.sigma = st.seed = st.ids = None
        if self.method == "smoothgrad":
            st.sigma = torch.tensor([self.noise * (self.hi - self.lo)], dtype=torch.float32, device=dev)
            st.seed = torch.zeros(1, dtype=torch.int64, device=dev)
            st.ids = torch.arange(N, dtype=torch.int64, device=dev)
        st.prologue, st.point = self._capture(st, self._prologue, self._iteration)

    def _run(self, x, labels, setup):
        x, labels, key = check_call(self.name, self.model, x, labels)
        st = self._graphed(key, x)
        setup(st)
        st.x.copy_(x)
        self._set_labels(st, labels)
        st.prologue.replay()
        for _ in range(st.alpha.numel()):
            st.point.replay()
        return st


class IntegratedGradients(_Attribution):
    """Integrated Gradients (Sundararajan et al., 2017) with `steps` trapezoid intervals (steps + 1 path points).  The
    captured graphs live on this object (deleting it frees them); a new x or baseline of a seen shape reuses them."""
    name, method = "IntegratedGradients", "ig"

    def __init__(self, model, steps=32, lo=-1.0, hi=1.0):
        if int(steps) < 1:
            raise ValueError(f"{self.name}: steps ({steps}) must be >= 1")
        super().__init__(model, lo, hi)
        self.steps = int(steps)

    def _tables(self):
        m = self.steps
        return [k / m for k in range(m + 1)], [0.5 / m if k in (0, m) else 1.0 / m for k in range(m + 1)]

    def __call__(self, x, labels=None, baseline=None):
        st = self._run(x, labels, lambda st: self._baseline(st, baseline, x))
        attr = st.attr.clone()
        f_x, f_b = st.f_x.clone(), st.f_b.clone()
        delta = attr.flatten(1).sum(1, dtype=torch.float64) - (f_x.double() - f_b.double())
        return {"attr": attr, "map": st.map.clone(), "target": st.target.clone(), "f_x": f_x, "f_baseline": f_b,
                "delta": delta}


class SmoothGrad(_Attribution):
    """SmoothGrad (Smilkov et al., 2017): the mean gradient of F over `draws` noisy copies x + sigma*eps, sigma =
    noise*(hi - lo).  SmoothGrad(draws=1, noise=0) is the vanilla gradient."""
    name, method = "SmoothGrad", "smoothgrad"

    def __init__(self, model, draws=16, noise=0.15, lo=-1.0, hi=1.0):
        if int(draws) < 1:
            raise ValueError(f"{self.name}: draws ({draws}) must be >= 1")
        if not float(noise) >= 0.0:
            raise ValueError(f"{self.name}: noise must be >= 0, got {noise}")
        super().__init__(model, lo, hi)
        self.draws, self.noise = int(draws), float(noise)

    def _tables(self):
        return [1.0] * self.draws, [1.0 / self.draws] * self.draws

    def __call__(self, x, labels=None, ids=None, seed=0):
        seed = L.seed_bits(seed, self.name)
        ids = L.require_ids(ids, x, self.name)

        def setup(st):
            st.seed.fill_(seed)
            if ids is None:
                torch.arange(st.ids.numel(), out=st.ids)
            else:
                st.ids.copy_(ids)

        st = self._run(x, labels, setup)
        return {"attr": st.attr.clone(), "map": st.map.clone(), "target": st.target.clone()}


class Faithfulness(_Explainer):
    """Deletion and insertion curves of an attribution map at `points` + 1 points, with their AUCs."""
    name = "Faithfulness"

    def __init__(self, model, points=16, lo=-1.0, hi=1.0):
        if int(points) < 1:
            raise ValueError(f"{self.name}: points ({points}) must be >= 1")
        super().__init__(model, lo, hi)
        self.points = int(points)

    def _prologue(self, st):
        self._target(st)
        st.j.zero_()

    def _point(self, st):
        ops.attrib_mask(st.x, st.b, st.rank, st.t, st.j, st.y_del, False)
        ops.attrib_mask(st.x, st.b, st.rank, st.t, st.j, st.y_ins, True)
        col = st.j.long()
        with self._autocast(st), torch.no_grad():
            for y, s in ((st.y_del, st.deletion), (st.y_ins, st.insertion)):
                p = objective(self.model(y)["cls_out"], st.target).exp()
                s.index_copy_(1, col, p[:, None])
        st.j.add_(1)

    def _state(self, st, x):
        self._new_state(st, x)
        N, C, H, W = x.shape
        dev, K = x.device, self.points
        st.b = torch.full_like(x, self.lo)
        st.rank = torch.zeros(N, H, W, dtype=torch.int32, device=dev)
        st.t = torch.tensor([j * H * W // K for j in range(K + 1)], dtype=torch.int32, device=dev)
        st.j = torch.zeros(1, dtype=torch.int32, device=dev)
        st.y_del, st.y_ins = torch.empty_like(x), torch.empty_like(x)
        st.deletion = torch.zeros(N, K + 1, device=dev)
        st.insertion = torch.zeros(N, K + 1, device=dev)
        st.prologue, st.point = self._capture(st, self._prologue, self._point)

    def __call__(self, x, amap, labels=None, baseline=None):
        x, labels, key = check_call(self.name, self.model, x, labels)
        N, _, H, W = x.shape
        if not torch.is_tensor(amap) or amap.shape != (N, H, W):
            raise ValueError(f"{self.name}: the map must be [N, H, W] = {(N, H, W)}, got "
                             f"{tuple(amap.shape) if torch.is_tensor(amap) else type(amap).__name__}")
        if not amap.is_cuda or amap.dtype != torch.float32 or amap.device != x.device:
            raise RuntimeError(f"{self.name}: the map must be an fp32 tensor on {x.device}")
        st = self._graphed(key, x)
        self._baseline(st, baseline, x)
        st.x.copy_(x)
        self._set_labels(st, labels)
        st.rank.copy_(ops.rank_desc(amap.detach().contiguous()))
        st.prologue.replay()
        for _ in range(self.points + 1):
            st.point.replay()
        d, i = st.deletion.clone(), st.insertion.clone()
        auc = lambda s: (s[:, :-1] + s[:, 1:]).sum(1) / (2 * self.points)       # noqa: E731
        return {"deletion": d, "insertion": i, "deletion_auc": auc(d), "insertion_auc": auc(i)}
