"""Fourier heat maps of the UniDefense detectors: accuracy and AUC under a Fourier-basis perturbation at each frequency
of a grid (after Yin et al., "A Fourier Perspective on Model Robustness in Computer Vision", NeurIPS 2019).

    hm = fourier.FourierHeatMap(model.eval(), eps=4.0, radius=15, stride=None, lo=-1.0, hi=1.0)
    r = hm(batches, seed=0)      # {"u", "v", "acc", "auc": [2R+1, R+1], "clean": {"acc", "auc", "n"}, "eps", "peak"}

At grid point (u, v) = (a*stride, b*stride), a = -R..R, b = 0..R, every sample gets x + r*eps*U_{u,v}, clamped to
[lo, hi]: U_{u,v} is the unit-norm cosine image whose 2-D spectrum sits at +-(u, v), and r = +-1 is drawn per sample
and channel, keyed by the sample id, the frequency and the seed (so sample i gets the same perturbation in any batch,
grid and rank).  eps is the L2 norm of the perturbation of each channel plane, in input units; "peak" is the
per-pixel amplitude eps*sqrt(2/(H*W)) at every frequency but DC and the Nyquist points.  U_{u,v} = U_{-u,-v}, so each
canonical frequency is evaluated once and its result fills every grid point that maps to it.  stride=None takes
floor(floor(min(H, W)/2) / R), so the grid reaches toward Nyquist (380^2, R = 15: stride 12, 481 frequencies).
Exact definitions: include/unidefense_b200.h (ud_fourier_perturb).

Two graphs are captured per input shape, autocast state and device and replayed (_evaluator.GraphedEvaluator): the
clean forward, then one frequency point (ud_fourier_perturb, a no_grad forward, the scores into row f of [F, N]
buffers, f += 1), replayed F times per batch.  Nothing synchronises with the host until the one read of the metrics
at the end.  The caller's torch.autocast context applies.
"""
import math

import torch

from . import _lib as L
from . import ops
from ._evaluator import GraphedEvaluator, p_fake, tally


def canonical(u, v, H, W):
    """The canonical (uu, vv) of the signed frequency (u, v) on an H x W image: the lexicographically smaller of
    (u mod H, v mod W) and ((-u) mod H, (-v) mod W)."""
    return min((u % H, v % W), ((-u) % H, (-v) % W))


def default_stride(H, W, radius):
    return (min(H, W) // 2) // radius


def grid(H, W, radius, stride):
    """-> (u [2R+1], v [R+1], the canonical frequencies [F] in first-seen order, index [2R+1][R+1] into them)."""
    u = [a * stride for a in range(-radius, radius + 1)]
    v = [b * stride for b in range(radius + 1)]
    table, slot, index = [], {}, []
    for uu in u:
        row = []
        for vv in v:
            c = canonical(uu, vv, H, W)
            if c not in slot:
                slot[c] = len(table)
                table.append(c)
            row.append(slot[c])
        index.append(row)
    return u, v, table, index


class FourierHeatMap(GraphedEvaluator):
    """Accuracy and AUC of a binary detector under Fourier-basis perturbations of L2 norm `eps` per channel plane.  The
    captured graphs live on this object (deleting it frees them); a new eps, seed or batch of a seen shape reuses them."""
    name = "FourierHeatMap"

    def __init__(self, model, eps, radius=15, stride=None, lo=-1.0, hi=1.0):
        if isinstance(radius, bool) or int(radius) != radius or int(radius) < 1:
            raise ValueError(f"{self.name}: radius must be an int >= 1, got {radius!r}")
        if stride is not None and (isinstance(stride, bool) or int(stride) != stride or int(stride) < 1):
            raise ValueError(f"{self.name}: stride must be None or an int >= 1, got {stride!r}")
        super().__init__(model, lo, hi)
        self.radius, self.stride = int(radius), None if stride is None else int(stride)
        self.eps = eps

    @property
    def eps(self):
        return self._eps

    @eps.setter
    def eps(self, value):
        value = float(value)
        if not (value >= 0.0 and math.isfinite(value)):
            raise ValueError(f"{self.name}: eps must be a finite float >= 0, got {value}")
        self._eps = value

    def _grid(self, H, W):
        R = self.radius
        s = default_stride(H, W, R) if self.stride is None else self.stride
        if s < 1:
            raise ValueError(f"{self.name}: a {H}x{W} image is too small for radius {R} (stride would be 0)")
        if s * R > H // 2 or s * R > W // 2:
            raise ValueError(f"{self.name}: stride*radius = {s}*{R} exceeds the Nyquist frequency of a {H}x{W} image "
                             f"({H // 2}, {W // 2})")
        return grid(H, W, R, s)

    def _prologue(self, st):
        with self._autocast(st), torch.no_grad():
            p, pred = p_fake(self.model(st.x)["cls_out"])
        st.p_clean.copy_(p)
        st.hit_clean.copy_(pred == st.labels)
        st.f.zero_()

    def _point(self, st):
        ops.fourier_perturb(st.x, st.y, st.freqs, st.f, st.eps, st.ids, st.seed, self.lo, self.hi)
        with self._autocast(st), torch.no_grad():
            p, pred = p_fake(self.model(st.y)["cls_out"])
        row = st.f.long()
        st.p.index_copy_(0, row, p[None])
        st.hit.index_copy_(0, row, (pred == st.labels)[None])
        st.f.add_(1)

    def _state(self, st, x, table):
        N, dev, F = x.shape[0], x.device, len(table)
        st.x, st.y = x.clone(), torch.empty_like(x)
        st.labels = torch.zeros(N, dtype=torch.long, device=dev)
        st.ids = torch.arange(N, dtype=torch.int64, device=dev)
        st.seed = torch.zeros(1, dtype=torch.int64, device=dev)
        st.eps = torch.zeros(1, device=dev)
        st.freqs = torch.tensor(table, dtype=torch.int32, device=dev)
        st.f = torch.zeros(1, dtype=torch.int32, device=dev)
        st.p = torch.zeros(F, N, device=dev)
        st.hit = torch.zeros(F, N, dtype=torch.bool, device=dev)
        st.p_clean = torch.zeros(N, device=dev)
        st.hit_clean = torch.zeros(N, dtype=torch.bool, device=dev)
        st.prologue, st.point = self._capture(st, self._prologue, self._point)

    def __call__(self, batches, seed=0):
        """batches yields (x, labels) or (x, labels, ids): x CUDA fp32 [N, C, H, W] of one C, H, W, labels {0 real,
        1 fake}, ids int64 [N] (default: the running sample index over the iterable).  The model must be in eval mode."""
        seed = L.seed_bits(seed, self.name)
        plane, g = None, None

        def score(x, labels, ids, key):
            nonlocal plane, g
            if plane is None:
                plane = tuple(x.shape[1:])
                g = self._grid(*plane[1:])
            elif tuple(x.shape[1:]) != plane:
                raise ValueError(f"{self.name}: every batch of a call must be [N, {', '.join(map(str, plane))}], "
                                 f"got {tuple(x.shape)}")
            st = self._graphed(key, x, g[2])
            st.x.copy_(x)
            st.labels.copy_(labels)
            st.ids.copy_(ids)
            st.eps.fill_(self.eps)
            st.seed.fill_(seed)
            st.prologue.replay()
            for _ in range(len(g[2])):
                st.point.replay()
            return torch.cat([st.p_clean[None], st.p]), torch.cat([st.hit_clean[None], st.hit])

        (acc, auc), n = tally(self.name, self.model, batches, score)
        index = torch.tensor(g[3])
        H, W = plane[1:]
        return {"u": torch.tensor(g[0], dtype=torch.int64), "v": torch.tensor(g[1], dtype=torch.int64),
                "acc": acc[1:][index], "auc": auc[1:][index],
                "clean": {"acc": float(acc[0]), "auc": float(auc[0]), "n": n},
                "eps": self.eps, "peak": self.eps * math.sqrt(2.0 / (H * W))}
