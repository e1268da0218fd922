"""PGD robustness-evaluation timings on the GPU: (1) ms per PGD iteration (forward, per-sample loss, d loss / dx, step)
as a hand-written eager torch loop against unidefense_b200.attack.PGD's graph replay, for UDEB4 @380^2 (N=32, N=8) and
UDR50 @256^2 (N=64), fp32 and under bf16 autocast; (2) ud_attack_step alone at 380^2, N=32 (L-inf, L2, select only)
with its algorithmic bytes and share of HBM bandwidth.

    python tools/attack_bench.py --out profiles/r05_attack_bench.json

Iteration times are CUDA-event means over --iters iterations after warm-up.  Kernel times are CUDA-event means over
--kernel-iters launches with the 126 MB L2 overwritten before every launch (inputs come from HBM) and every sample set
to improve (x_best is written: the most bytes).  Bytes are what the algorithm must move; "HBM share" = bytes / time /
7.7 TB/s (data-sheet HBM3e bandwidth of one B200).
"""
import argparse
import json
import math
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from input_grad_bench import HBM, gpu_info, timeit  # noqa: E402

CONFIGS = (("UDEB4", dict(extractor="efficientnet-b4", num_classes=2), 32, 380),
           ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2), 8, 380),
           ("UDR50", dict(extractor="resnet50", num_classes=2), 64, 256))


def per_iteration(iters, flush):
    from oracle import attack as A
    from unidefense_b200.attack import PGD
    from unidefense_b200.model import load_model
    rows = []
    for name, kw, N, R in CONFIGS:
        torch.manual_seed(0)
        model = load_model(name)(**kw).cuda().eval()
        x0 = torch.rand(N, 3, R, R, device="cuda") * 2 - 1
        labels = torch.arange(N, device="cuda") % 2
        eps = torch.full((N,), 16 / 255, device="cuda")
        alpha = eps / 4
        for amp in (None, torch.bfloat16):
            ctx = (lambda: torch.autocast("cuda", dtype=amp)) if amp else (lambda: torch.autocast("cuda", enabled=False))
            x_adv, x_best = x0.clone(), x0.clone()
            best = torch.full((N,), -math.inf, device="cuda")

            def eager():                     # forward, autograd.grad, then torch elementwise select + step + projection
                xin = x_adv.detach().requires_grad_()
                with ctx():
                    loss = F.cross_entropy(model(xin)["cls_out"].float(), labels, reduction="none")
                g, = torch.autograd.grad(loss.sum(), xin)
                with torch.no_grad():
                    nb, nx, _ = A.select(loss, best, x_adv, x_best)
                    best.copy_(nb)
                    x_best.copy_(nx)
                    x_adv.copy_(A.linf_step(x0, x_adv, g, eps, alpha, -1.0, 1.0))

            eager_ms = timeit(eager, iters, flush)
            atk = PGD(model, steps=1)
            with ctx():
                atk(x0, labels)              # captures
            st, = atk._graphs.values()
            graph_ms = timeit(st.step.replay, iters, flush)
            rows.append({"model": name, "N": N, "R": R, "autocast": "bf16" if amp else "fp32",
                         "eager_ms_per_iteration": eager_ms, "graph_ms_per_iteration": graph_ms,
                         "speedup": eager_ms / graph_ms})
            print(json.dumps(rows[-1]), flush=True)
            del atk, st
            torch.cuda.empty_cache()
        del model
        torch.cuda.empty_cache()
    return rows


def step_kernel(iters, flush):
    from unidefense_b200 import ops
    N, R = 32, 380
    P = 3 * R * R
    g = torch.Generator(device="cuda").manual_seed(0)
    x0 = torch.rand(N, 3, R, R, device="cuda", generator=g) * 2 - 1
    x_adv = (x0 + 0.01 * torch.randn(N, 3, R, R, device="cuda", generator=g)).clamp(-1, 1)
    grad = torch.randn(N, 3, R, R, device="cuda", generator=g)
    x_best = torch.empty_like(x0)
    loss = torch.zeros(N, device="cuda")
    best = torch.empty(N, device="cuda")
    eps = torch.full((N,), 16 / 255, device="cuda")
    alpha = eps / 4
    img = N * P * 4
    rows = []
    for label, norm, gg, nbytes, note in (
            ("linf", "linf", grad, 5 * img, "reads x0, x_adv, g; writes x_adv, x_best"),
            ("l2", "l2", grad, 9 * img, "g-norm pass reads g; d-norm pass reads x0, x_adv, g; apply pass as L-inf"),
            ("select only", "linf", None, 2 * img, "reads x_adv; writes x_best")):
        def call():
            ops.attack_step(x0, x_adv, gg, loss, best, x_best, eps, alpha, -1.0, 1.0, norm)
        for _ in range(3):
            best.fill_(-math.inf)
            call()
        torch.cuda.synchronize()
        tot = 0.0
        for _ in range(iters):
            best.fill_(-math.inf)            # every sample improves
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        ms = tot / iters
        rows.append({"call": f"ud_attack_step ({label})", "N": N, "R": R, "us": ms * 1e3, "bytes": nbytes,
                     "GB_per_s": nbytes / ms / 1e6, "hbm_share": nbytes / (ms * 1e-3) / HBM, "note": note})
        print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "attack_bench.json"))
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--kernel-iters", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attack_bench.py measures on the GPU; no CUDA device found")
    torch.backends.cudnn.benchmark = False
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2
    res = {"gpu": gpu_info(), "step_kernel_380_n32": step_kernel(args.kernel_iters, flush),
           "pgd_iteration": per_iteration(args.iters, flush)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
