"""Corruption-robustness timings on the GPU: (1) ud_corrupt per kind and severity at 380², N=32 and 256², N=64, with
algorithmic bytes and share of HBM bandwidth; (2) the same corruptions on the host through OpenCV / numpy (the path
users have without these kernels), images/s single-threaded and on all cores; (3) corrupt.evaluate on UDEB4 at 380²,
N=32 under bf16 autocast, ms per batch split into corruption and forward.

    python tools/corrupt_bench.py --out profiles/r06_corrupt_bench.json

Kernel times are CUDA-event means over --kernel-iters calls with the 126 MB L2 overwritten before every call.  Bytes
are what the algorithm must move: the input read and the output written once (block adds its squares, jpeg its decoded
planes written and read back through the workspace); halo re-reads are not counted.  "HBM share" = bytes / time /
7.7 TB/s (data-sheet HBM3e bandwidth of one B200).
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from input_grad_bench import HBM, gpu_info, timeit  # noqa: E402


def kernel_rows(iters, flush):
    from oracle import corrupt as C
    from unidefense_b200 import corrupt
    rows = []
    for N, R in ((32, 380), (64, 256)):
        x = torch.from_numpy(C.test_images(N, R, R, seed=0)).cuda()
        ids = torch.arange(N, device="cuda")
        img = N * 3 * R * R * 4
        for kind in corrupt.KINDS:
            for sev in range(1, 6):
                p = corrupt.LEVELS[kind][sev - 1]
                nbytes = 2 * img
                if kind == "block":
                    nbytes += N * p * 64 * 3 * 4
                elif kind == "jpeg":
                    nbytes += 2 * N * (R * R + 2 * ((R + 1) // 2) ** 2) * 4
                ms = timeit(lambda: corrupt.apply(x, kind, sev, ids=ids), iters, flush)
                rows.append({"kind": kind, "severity": sev, "param": p, "N": N, "R": R, "us": ms * 1e3,
                             "bytes": nbytes, "hbm_share": nbytes / (ms * 1e-3) / HBM})
                print(json.dumps(rows[-1]), flush=True)
    return rows


# ---- host baseline: OpenCV / numpy on uint8 HxWx3 RGB frames --------------------------------------------------------
def _host(img, kind, p, rng):
    import cv2
    if kind == "saturation":
        ycc = cv2.cvtColor(img, cv2.COLOR_RGB2YCrCb).astype(np.float32)
        ycc[..., 1:] = 128 + (ycc[..., 1:] - 128) * p
        return cv2.cvtColor(np.clip(np.rint(ycc), 0, 255).astype(np.uint8), cv2.COLOR_YCrCb2RGB)
    if kind == "contrast":
        return cv2.convertScaleAbs(img, alpha=p)
    if kind == "block":
        out = img.copy()
        H, W = img.shape[:2]
        for r, c in zip(rng.integers(0, H - 7, p), rng.integers(0, W - 7, p)):
            out[r:r + 8, c:c + 8] = 128
        return out
    if kind == "noise":
        ycc = cv2.cvtColor(img, cv2.COLOR_RGB2YCrCb).astype(np.float32) / 255
        ycc += np.sqrt(p) * rng.standard_normal(ycc.shape, dtype=np.float32)
        return cv2.cvtColor(np.clip(ycc * 255, 0, 255).astype(np.uint8), cv2.COLOR_YCrCb2RGB)
    if kind == "blur":
        return cv2.GaussianBlur(img, (p, p), p / 6)
    if kind == "pixelate":
        H, W = img.shape[:2]
        small = cv2.resize(img, ((W + p - 1) // p, (H + p - 1) // p), interpolation=cv2.INTER_AREA)
        return cv2.resize(small, (W, H), interpolation=cv2.INTER_NEAREST)
    ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, p])
    return cv2.imdecode(enc, cv2.IMREAD_COLOR)


def _host_work(args):
    import cv2
    cv2.setNumThreads(1)
    kind, p, R, n = args
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (R, R, 3), dtype=np.uint8)
    for _ in range(n):
        _host(img, kind, p, rng)
    return n


def host_rows(R=380, per_worker=64):
    from unidefense_b200 import corrupt
    workers = os.cpu_count()
    rows = []
    with mp.get_context("spawn").Pool(workers) as pool:
        for kind in corrupt.KINDS:
            p = corrupt.LEVELS[kind][2]
            _host_work((kind, p, R, 4))
            t = time.perf_counter()
            _host_work((kind, p, R, per_worker))
            single = per_worker / (time.perf_counter() - t)
            pool.map(_host_work, [(kind, p, R, 2)] * workers)
            t = time.perf_counter()
            n = sum(pool.map(_host_work, [(kind, p, R, per_worker)] * workers))
            allc = n / (time.perf_counter() - t)
            rows.append({"kind": kind, "severity": 3, "param": p, "R": R, "img_per_s_1_thread": single,
                         "img_per_s_all_cores": allc, "cores": workers})
            print(json.dumps(rows[-1]), flush=True)
    return rows


def evaluate_split(iters):
    from oracle import corrupt as C
    from unidefense_b200 import corrupt
    from unidefense_b200.model import load_model
    N, R = 32, 380
    torch.manual_seed(0)
    model = load_model("UDEB4")(extractor="efficientnet-b4", num_classes=2).cuda().eval()
    x = torch.from_numpy(C.test_images(N, R, R, seed=0)).cuda()
    labels = torch.arange(N, device="cuda") % 2
    ids = torch.arange(N, device="cuda")
    keys = [(k, s) for k in corrupt.KINDS for s in range(1, 6)]
    ys = [corrupt.apply(x, k, s, ids=ids) for k, s in keys]

    def ev(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    with torch.autocast("cuda", dtype=torch.bfloat16):
        total = ev(lambda: corrupt.evaluate(model, [(x, labels, ids)]))
        with torch.no_grad():
            fwd = ev(lambda: [model(v)["cls_out"] for v in [x] + ys])
        corr = ev(lambda: [corrupt.apply(x, k, s, ids=ids) for k, s in keys])
    row = {"model": "UDEB4", "N": N, "R": R, "autocast": "bf16", "forwards_per_batch": 1 + len(keys),
           "corruptions_per_batch": len(keys), "evaluate_ms_per_batch": total, "corruption_ms": corr,
           "forward_ms": fwd, "corruption_share": corr / total}
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "corrupt_bench.json"))
    ap.add_argument("--kernel-iters", type=int, default=50)
    ap.add_argument("--iters", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("corrupt_bench.py measures on the GPU; no CUDA device found")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2
    res = {"gpu": gpu_info(), "kernels": kernel_rows(args.kernel_iters, flush), "host": host_rows(),
           "evaluate": evaluate_split(args.iters)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["evaluate"], indent=1))


if __name__ == "__main__":
    main()
