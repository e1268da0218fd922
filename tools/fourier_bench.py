"""Fourier heat-map timings on the GPU: (a) ud_fourier_perturb alone at 380^2, N=32, with its bytes and share of HBM
bandwidth; (b) ms per frequency point (perturb, no_grad forward, scores) as a hand-written eager torch loop against
unidefense_b200.fourier's graph replay, UDEB4 @380^2 under bf16 autocast at N=32 and N=8; (c) one whole
FourierHeatMap call at the default grid (radius 15: 31 x 16 grid points, 481 frequencies) on one N=32 batch, with the
map's shape and the equality of the mirror pairs of its v = 0 column.

    python tools/fourier_bench.py --out profiles/r10_fourier_bench.json

Times are CUDA-event means after warm-up.  (a) and (b) overwrite the 126 MB L2 before every timed launch (inputs come
from HBM); "HBM share" = bytes / time / 7.7 TB/s (data-sheet HBM3e bandwidth of one B200).  (c) is timed from the
host around the call, which ends in its one device-to-host read, after a first call that captured the graphs.
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from input_grad_bench import HBM, gpu_info, timeit  # noqa: E402

R = 380


def _inputs(N):
    g = torch.Generator(device="cuda").manual_seed(N)
    x = torch.rand(N, 3, R, R, device="cuda", generator=g) * 2 - 1
    labels = torch.arange(N, device="cuda") % 2
    return x, labels


def kernel(iters, flush):
    from unidefense_b200 import ops
    from unidefense_b200.fourier import grid
    N = 32
    x, _ = _inputs(N)
    y = torch.empty_like(x)
    _, _, table, _ = grid(R, R, 15, 12)
    freqs = torch.tensor(table, dtype=torch.int32, device="cuda")
    f = torch.tensor([100], dtype=torch.int32, device="cuda")
    eps = torch.tensor([4.0], device="cuda")
    seed = torch.zeros(1, dtype=torch.int64, device="cuda")
    nbytes = 2 * N * 3 * R * R * 4
    ms = timeit(lambda: ops.fourier_perturb(x, y, freqs, f, eps, None, seed, -1.0, 1.0), iters, flush)
    row = {"call": "ud_fourier_perturb", "N": N, "R": R, "frequency": list(table[100]), "us": ms * 1e3,
           "bytes": nbytes, "GB_per_s": nbytes / ms / 1e6, "hbm_share": nbytes / (ms * 1e-3) / HBM,
           "note": "reads x, writes y (2*N*3*H*W*4 bytes)"}
    print(json.dumps(row), flush=True)
    return [row]


def _model():
    from unidefense_b200.model import load_model
    torch.manual_seed(0)
    return load_model("UDEB4")(extractor="efficientnet-b4", num_classes=2).cuda().eval()


def per_point(iters, flush):
    from unidefense_b200 import ops
    from unidefense_b200._evaluator import p_fake
    from unidefense_b200.fourier import FourierHeatMap
    model = _model()
    rows = []
    for N in (32, 8):
        x, labels = _inputs(N)
        hm = FourierHeatMap(model, 4.0, radius=2)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            hm([(x, labels)])                   # captures
            st, = hm._graphs.values()
            y = torch.empty_like(x)
            p_buf = torch.empty(N, device="cuda")

            def eager():                        # the kernel, a no_grad forward, the scores
                ops.fourier_perturb(x, y, st.freqs, st.f, st.eps, None, st.seed, -1.0, 1.0)
                with torch.no_grad():
                    p, pred = p_fake(model(y)["cls_out"])
                p_buf.copy_(p)

            def replay():
                st.f.fill_(1)
                st.point.replay()

            st.f.fill_(1)
            eager_ms = timeit(eager, iters, flush)
            graph_ms = timeit(replay, iters, flush)
        rows.append({"model": "UDEB4", "N": N, "R": R, "autocast": "bf16", "eager_ms_per_point": eager_ms,
                     "graph_ms_per_point": graph_ms, "speedup": eager_ms / graph_ms})
        print(json.dumps(rows[-1]), flush=True)
        del hm, st
        torch.cuda.empty_cache()
    return rows


def whole_call(call_iters):
    from unidefense_b200.fourier import FourierHeatMap
    model = _model()
    N = 32
    x, labels = _inputs(N)
    hm = FourierHeatMap(model, 4.0)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        t0 = time.perf_counter()
        r = hm([(x, labels)], seed=0)
        first_s = time.perf_counter() - t0
        times = []
        for _ in range(call_iters):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = hm([(x, labels)], seed=0)
            times.append(time.perf_counter() - t0)
    F = len(next(iter(hm._graphs.values())).freqs)
    ms = 1e3 * sum(times) / len(times)
    acc = r["acc"]
    mirror = all(float(acc[i, 0]) == float(acc[acc.shape[0] - 1 - i, 0]) for i in range(acc.shape[0]))
    row = {"call": "FourierHeatMap(eps=4.0) default grid", "model": "UDEB4", "N": N, "R": R, "autocast": "bf16",
           "grid": list(acc.shape), "frequencies": F, "forwards": F + 1, "ms": ms, "ms_per_forward": ms / (F + 1),
           "first_call_s_with_capture": first_s, "v0_mirror_pairs_equal": mirror, "clean": r["clean"],
           "peak": r["peak"], "acc_min": float(acc.min()), "acc_max": float(acc.max())}
    print(json.dumps(row), flush=True)
    return [row]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fourier_bench.json"))
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--call-iters", type=int, default=1)
    ap.add_argument("--kernel-iters", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fourier_bench.py measures on the GPU; no CUDA device found")
    torch.backends.cudnn.benchmark = False
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2
    res = {"gpu": gpu_info(), "kernel_380_n32": kernel(args.kernel_iters, flush),
           "per_point": per_point(args.iters, flush), "whole_call": whole_call(args.call_iters)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
