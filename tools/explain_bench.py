"""Attribution timings on the GPU: (1) ud_attrib_step (IG and SmoothGrad middle steps, the IG last step), ud_attrib_mask
and ud_rank_desc alone at 380^2, N=32, with their bytes and share of HBM bandwidth; (2) ms per IG iteration (forward,
F, d F / dx, step) as a hand-written eager torch loop against unidefense_b200.explain's graph replay, UDEB4 @380^2 under
bf16 autocast at N=32 and N=8; (3) whole-call times of IntegratedGradients (steps=32), SmoothGrad (draws=16) and
Faithfulness (points=16) on UDEB4 @380^2, N=32, bf16.

    python tools/explain_bench.py --out profiles/r09_explain_bench.json

Times are CUDA-event means after warm-up.  Kernel times overwrite the 126 MB L2 before every launch (inputs come from
HBM), except ud_rank_desc's per-plane sort workspace, which the sort itself keeps in L2.  Bytes are what each kernel
reads and writes in HBM; "HBM share" = bytes / time / 7.7 TB/s (data-sheet HBM3e bandwidth of one B200).
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from input_grad_bench import HBM, gpu_info, timeit  # noqa: E402


def kernels(iters, flush):
    from unidefense_b200 import ops
    N, R = 32, 380
    HW = R * R
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(N, 3, R, R, device="cuda", generator=g) * 2 - 1
    b = torch.rand(N, 3, R, R, device="cuda", generator=g) * 0.1 - 1
    grad = torch.randn(N, 3, R, R, device="cuda", generator=g)
    acc, p, attr = torch.zeros_like(x), torch.empty_like(x), torch.empty_like(x)
    amap = torch.rand(N, R, R, device="cuda", generator=g)
    img = N * 3 * HW * 4
    plane = N * HW * 4
    S = 33
    alpha = torch.linspace(0, 1, S, device="cuda")
    w = torch.full((S,), 1 / 32, device="cuda")
    sigma = torch.tensor([0.3], device="cuda")
    seed = torch.zeros(1, dtype=torch.int64, device="cuda")
    mid = torch.tensor([5], dtype=torch.int32, device="cuda")
    last = torch.tensor([S - 1], dtype=torch.int32, device="cuda")
    rank = ops.rank_desc(amap)
    t = torch.tensor([j * HW // 16 for j in range(17)], dtype=torch.int32, device="cuda")
    j = torch.tensor([8], dtype=torch.int32, device="cuda")
    y = torch.empty_like(x)
    rows = []
    for label, fn, nbytes, note in (
            ("ud_attrib_step (IG, middle step, tensor baseline)",
             lambda: ops.attrib_step(x, b, grad, acc, p, attr, amap, mid, alpha, w, "ig"), 6 * img,
             "reads x, b, g, acc; writes acc, p; the map launch exits at once"),
            ("ud_attrib_step (SmoothGrad, middle step)",
             lambda: ops.attrib_step(x, 0.0, grad, acc, p, attr, amap, mid, alpha, w, "smoothgrad", sigma, None, seed),
             5 * img, "reads x, g, acc; writes acc, p (Philox noise)"),
            ("ud_attrib_step (IG, last step)",
             lambda: ops.attrib_step(x, b, grad, acc, p, attr, amap, last, alpha, w, "ig"), 5 * img + img + plane,
             "reads x, b, g, acc; writes attr; map launch reads attr, writes map"),
            ("ud_attrib_mask (deletion, tensor baseline)",
             lambda: ops.attrib_mask(x, b, rank, t, j, y, False), 2 * img + plane,
             "reads rank and, per element, x or b; writes y"),
            ("ud_rank_desc", lambda: ops.rank_desc(amap), 2 * plane,
             "reads the map, writes rank; the 16 B/pixel sort workspace (74 MB) stays in L2")):
        ms = timeit(fn, iters, flush)
        rows.append({"call": label, "N": N, "R": R, "us": ms * 1e3, "bytes": nbytes, "GB_per_s": nbytes / ms / 1e6,
                     "hbm_share": nbytes / (ms * 1e-3) / HBM, "note": note})
        print(json.dumps(rows[-1]), flush=True)
    return rows


def _model():
    from unidefense_b200.model import load_model
    torch.manual_seed(0)
    return load_model("UDEB4")(extractor="efficientnet-b4", num_classes=2).cuda().eval()


def per_iteration(iters, flush):
    from oracle import explain as E
    from unidefense_b200.explain import IntegratedGradients
    model = _model()
    rows = []
    for N in (32, 8):
        R = 380
        x = torch.rand(N, 3, R, R, device="cuda") * 2 - 1
        b = torch.full_like(x, -1.0)
        acc, p = torch.zeros_like(x), x.clone()
        target = torch.arange(N, device="cuda") % 2
        with torch.autocast("cuda", dtype=torch.bfloat16):
            def eager():                     # forward, autograd.grad, then the torch accumulate + next point
                xin = p.detach().requires_grad_()
                f = E.objective(model(xin)["cls_out"].float(), target)
                g, = torch.autograd.grad(f.sum(), xin)
                with torch.no_grad():
                    acc.copy_(E.accumulate(acc, 1 / 32, g))
                    p.copy_(E.path_point(x, b, 0.5))
            eager_ms = timeit(eager, iters, flush)
            ig = IntegratedGradients(model, steps=32)
            ig(x)                            # captures
            st, = ig._graphs.values()
            def replay():                    # from a middle step: the step kernel runs, the map launch exits
                st.k.fill_(5)
                st.point.replay()
            graph_ms = timeit(replay, iters, flush)
        rows.append({"model": "UDEB4", "N": N, "R": R, "autocast": "bf16", "eager_ms_per_iteration": eager_ms,
                     "graph_ms_per_iteration": graph_ms, "speedup": eager_ms / graph_ms})
        print(json.dumps(rows[-1]), flush=True)
        del ig, st
        torch.cuda.empty_cache()
    return rows


def whole_calls(iters, flush):
    from unidefense_b200.explain import Faithfulness, IntegratedGradients, SmoothGrad
    model = _model()
    N, R = 32, 380
    x = torch.rand(N, 3, R, R, device="cuda") * 2 - 1
    rows = []
    with torch.autocast("cuda", dtype=torch.bfloat16):
        ig, sg, fa = IntegratedGradients(model, steps=32), SmoothGrad(model, draws=16), Faithfulness(model, points=16)
        amap = ig(x)["map"]
        for label, fn in (("IntegratedGradients(steps=32)", lambda: ig(x)), ("SmoothGrad(draws=16)", lambda: sg(x)),
                          ("Faithfulness(points=16)", lambda: fa(x, amap))):
            ms = timeit(fn, iters, flush)
            rows.append({"call": label, "model": "UDEB4", "N": N, "R": R, "autocast": "bf16", "ms": ms})
            print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "explain_bench.json"))
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--call-iters", type=int, default=3)
    ap.add_argument("--kernel-iters", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("explain_bench.py measures on the GPU; no CUDA device found")
    torch.backends.cudnn.benchmark = False
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2
    res = {"gpu": gpu_info(), "kernels_380_n32": kernels(args.kernel_iters, flush),
           "ig_iteration": per_iteration(args.iters, flush), "whole_call": whole_calls(args.call_iters, flush)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
