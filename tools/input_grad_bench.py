"""Input-gradient timings on the GPU: (1) the kernels that carry d/dx (UDEB4 380^2, N=32) with their algorithmic bytes
and share of HBM bandwidth, next to the training-path kernels they extend; (2) one attack step (eval, frozen
parameters, forward + d softmax(cls_out)[:,0].sum() / dx) for UDEB4@380 N=32 and UDR50@256 N=64; (3) the isolated
recon-path input gradient (error maps -> dynamic filters -> fuse, reconstruction tail; forward + d loss / dx), ours
against the stock-torch op sequence of tools/torch_bar.py under autograd.

    python tools/input_grad_bench.py --out profiles/input_grad_bench.json

Kernel and step times are CUDA-event means over --iters launches after warm-up, with the 126 MB L2 overwritten
before every timed launch (so a kernel's inputs come from HBM).  Bytes are what the algorithm must move, computed from
the shapes below; "HBM share" = bytes / time / 7.7 TB/s (data-sheet HBM3e bandwidth of one B200).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

HBM = 7.7e12


def timeit(fn, iters, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / iters


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}


def kernels(iters, flush):
    from unidefense_b200 import _lib as L
    lib, dev, s = L.lib(), "cuda", L.stream()
    N, C, h, R, he = 32, 3, 192, 380, 12
    g = torch.Generator().manual_seed(0)
    dec = torch.tanh(torch.randn(N, C, h, h, generator=g)).to(dev)
    x = (torch.rand(N, C, R, R, generator=g) * 2 - 1).to(dev)
    rows = []

    def row(name, fn, nbytes, note=""):
        ms = timeit(fn, iters, flush)
        rows.append({"kernel": name, "ms": ms, "bytes": nbytes, "GB_per_s": nbytes / ms / 1e6,
                     "hbm_share": nbytes / (ms * 1e-3) / HBM, "note": note})

    # recon tail backward: training path (g_dec) vs + g_x vs g_x alone
    signs = torch.empty(lib.ud_recon_tail_signs_bytes(N, C, R, R), dtype=torch.uint8, device=dev)
    rec, sp, fr = torch.empty_like(x), torch.empty(N, device=dev), torch.empty(N, device=dev)
    nws = lib.ud_recon_tail_workspace_bytes(N, C, h, h, R, R)
    ws = L.workspace(nws, x.device)
    L.check(lib.ud_recon_tail_fwd(L.ptr(dec), L.ptr(x), L.ptr(rec), L.ptr(sp), L.ptr(fr), L.ptr(signs), L.ptr(ws), nws,
                                  N, C, h, h, R, R, 1, s))
    gs, gf = torch.full((N,), 0.1, device=dev), torch.ones(N, device=dev)
    g_dec, g_x = torch.empty_like(dec), torch.empty_like(x)
    img, small, sb = N * C * R * R * 4, N * C * h * h * 4, signs.numel()
    row("recon_tail_bwd (g_dec)", lambda: L.check(lib.ud_recon_tail_bwd(
        L.ptr(dec), L.ptr(x), L.ptr(signs), L.ptr(gs), L.ptr(gf), L.ptr(g_dec), None, L.ptr(ws), nws, N, C, h, h, R, R, 1,
        s)), small + img + sb + small, "reads dec, x, signs; writes g_dec")
    row("recon_tail_bwd (g_dec + g_x)", lambda: L.check(lib.ud_recon_tail_bwd(
        L.ptr(dec), L.ptr(x), L.ptr(signs), L.ptr(gs), L.ptr(gf), L.ptr(g_dec), L.ptr(g_x), L.ptr(ws), nws, N, C, h, h, R,
        R, 1, s)), small + img + sb + small + img, "+ 3R^2*4 B written per sample")
    row("recon_tail_bwd (g_x only)", lambda: L.check(lib.ud_recon_tail_bwd(
        L.ptr(dec), L.ptr(x), L.ptr(signs), L.ptr(gs), L.ptr(gf), None, L.ptr(g_x), L.ptr(ws), nws, N, C, h, h, R, R, 1,
        s)), small + img + sb + img, "dec detached")
    # error maps -> x
    pred = torch.tanh(torch.randn(N, C, h, h, generator=g)).to(dev)
    gsd = torch.randn(N, C, he, he, generator=g).to(dev)
    gfd = torch.randn(N, 2 * C, he, he // 2 + 1, generator=g).to(dev)
    taps = 2 * 4 * N * C * he * he * 4          # 4 bilinear taps of pred and of x per small pixel
    row("attn_prep_bwd 380->12", lambda: L.check(lib.ud_attn_prep_bwd(
        L.ptr(pred), L.ptr(x), L.ptr(gsd), L.ptr(gfd), L.ptr(g_x), N, C, h, h, R, R, he, he, 1, s)),
        taps + gsd.numel() * 4 + gfd.numel() * 4 + img, "writes the dense g_x once")
    # dynamic filters at UDEB4's attention (freq: 544 ch @ 12x7, D=6; spatial: 272 ch @ 12x12, D=3)
    for kind, Cp, hw, D in (("freq", 544, 12 * 7, 6), ("spat", 272, 12 * 12, 3)):
        proj = torch.randn(N, Cp, hw, device=dev)
        xx = torch.randn(N, Cp, hw, device=dev)
        diff = torch.rand(N, D, hw, device=dev)
        mean, rstd = torch.zeros(Cp, device=dev), torch.ones(Cp, device=dev)
        gam, bet = torch.ones(Cp, device=dev), torch.zeros(Cp, device=dev)
        w2 = torch.randn(2 + D, device=dev)
        mask, out = torch.empty(N, hw, device=dev), torch.empty_like(xx)
        pm, px, am = torch.empty(N, hw, device=dev), torch.empty(N, hw, device=dev), torch.empty(N, hw, dtype=torch.int32,
                                                                                              device=dev)
        L.check(lib.ud_dyfi_mask_fwd(L.ptr(proj), L.ptr(mean), L.ptr(rstd), L.ptr(gam), L.ptr(bet), L.ptr(diff),
                                     L.ptr(w2), L.ptr(xx), L.ptr(mask), L.ptr(out), L.ptr(pm), L.ptr(px), L.ptr(am), N, Cp,
                                     D, Cp, hw, 2, s))
        go, gxx, dz, gw2, gd = torch.randn_like(xx), torch.empty_like(xx), torch.empty_like(proj), torch.empty(
            2 + D, device=dev), torch.empty_like(diff)
        wsd = L.workspace(lib.ud_dyfi_mask_bwd_workspace_bytes(N, hw), x.device)
        base = (3 * proj.numel() + 3 * xx.numel() + 4 * N * hw + D * N * hw) * 4
        row(f"dyfi_mask_bwd ({kind})", lambda: L.check(lib.ud_dyfi_mask_bwd(
            L.ptr(proj), L.ptr(mean), L.ptr(rstd), L.ptr(gam), L.ptr(bet), L.ptr(diff), L.ptr(w2), L.ptr(xx), L.ptr(mask),
            L.ptr(pm), L.ptr(px), L.ptr(am), None, L.ptr(go), L.ptr(gxx), L.ptr(dz), L.ptr(gw2), None, L.ptr(wsd),
            wsd.numel(), N, Cp, D, Cp, hw, 2, s)), base, "training path")
        row(f"dyfi_mask_bwd ({kind}, + g_diff)", lambda: L.check(lib.ud_dyfi_mask_bwd(
            L.ptr(proj), L.ptr(mean), L.ptr(rstd), L.ptr(gam), L.ptr(bet), L.ptr(diff), L.ptr(w2), L.ptr(xx), L.ptr(mask),
            L.ptr(pm), L.ptr(px), L.ptr(am), None, L.ptr(go), L.ptr(gxx), L.ptr(dz), L.ptr(gw2), L.ptr(gd), L.ptr(wsd),
            wsd.numel(), N, Cp, D, Cp, hw, 2, s)), base + gd.numel() * 4, "+ D*HW*4 B written per sample")
    gy = torch.randn_like(x)
    row("gaussian_blur5_bwd 380", lambda: L.check(lib.ud_gaussian_blur5_bwd(L.ptr(gy), L.ptr(g_x), N * C, R, R, s)),
        2 * img)
    row("downscale_nearest_bwd 380", lambda: L.check(lib.ud_downscale_nearest_bwd(L.ptr(gy), L.ptr(g_x), N * C, R, R,
                                                                                   0.75, s)), 2 * img)
    return rows


def attack_steps(iters, flush):
    from unidefense_b200.model import load_model
    out = []
    for name, kw, N, R in (("UDEB4", dict(extractor="efficientnet-b4", num_classes=2), 32, 380),
                           ("UDR50", dict(extractor="resnet50", num_classes=2), 64, 256)):
        torch.manual_seed(0)
        model = load_model(name)(**kw).cuda().eval().requires_grad_(False)
        x = (torch.rand(N, 3, R, R, device="cuda") * 2 - 1).requires_grad_()

        def step():
            score = torch.softmax(model(x)["cls_out"], dim=1)[:, 0].sum()
            return torch.autograd.grad(score, x)[0]

        def fwd():
            with torch.no_grad():
                return model(x)["cls_out"]

        out.append({"model": name, "N": N, "R": R, "attack_step_ms": timeit(step, iters, flush),
                    "eval_forward_ms": timeit(fwd, iters, flush)})
        del model
        torch.cuda.empty_cache()
    return out


def recon_path(iters, flush):
    import torch_bar as TB
    from unidefense_b200 import ops
    from unidefense_b200.model import load_model
    N, C, h, R, E, he = 32, 3, 192, 380, 272, 12
    g = torch.Generator().manual_seed(1)
    dec = torch.tanh(torch.randn(N, C, h, h, generator=g)).cuda()
    emb = torch.randn(N, E, he, he, generator=g).cuda()
    x0 = (torch.rand(N, C, R, R, generator=g) * 2 - 1).cuda()
    r_att = torch.randn(N, E, he, he, generator=g).cuda()
    torch.manual_seed(0)
    model = load_model("UDEB4")(extractor="efficientnet-b4", num_classes=2).cuda().train()
    p = TB.attention_params(E, "cuda")
    x = x0.clone().requires_grad_()

    def loss_of(att_out, fmask, smask, spatial, freq):
        return (0.1 * fmask.mean() + 0.1 * smask.mean() + 0.1 * spatial.mean() + freq.mean() + (att_out * r_att).sum())

    def ours():
        att = model.attention(dec, x, emb)
        _, sp, fr = ops.recon_tail(dec, x)
        return torch.autograd.grad(loss_of(att["out"], att["freq_mask"], att["spat_mask"], sp, fr), x)[0]

    def stock():
        a, fm, sm = TB.attention(dec, x, emb, p, "swish")
        _, sp, fr = TB.recon_tail(dec, x)
        return torch.autograd.grad(loss_of(a, fm, sm, sp, fr), x)[0]

    return {"shape": f"UDEB4 attention + recon tail, N={N}, x {R}^2, dec {h}^2, emb {E}x{he}^2",
            "ours_ms": timeit(ours, iters, flush), "stock_torch_ms": timeit(stock, iters, flush)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "input_grad_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("input_grad_bench.py measures on the GPU; no CUDA device found")
    torch.backends.cudnn.benchmark = False
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2
    res = {"gpu": gpu_info(), "kernels_udeb4_380_n32": kernels(args.iters, flush),
           "attack_step": attack_steps(args.iters, flush), "recon_path_x_grad": recon_path(args.iters, flush)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
