#!/usr/bin/env python3
"""Benchmark of the UniDefense dual-space reconstruction path on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 10 --warmup 3                    # our arm, 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W     # N GPUs, one rank per GPU (NCCL)
    python bench.py --impl reference --steps 3 --warmup 1             # reference arm: CPU port on the host cores
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs D   # + the last timed step's outputs as D/*.npy

A "step" is one training step of the drop-in UniDefenseModelEb4 (EfficientNet-B4, 380x380, per-GPU
batch 32, bf16 autocast + channels_last for the stock-torch backbone and dense convs, fp32 hot-path kernels)
on synthetic face tensors: forward, the engine's first-pass loss (engine/abstract_engine.py:215-267), backward
(+ NCCL gradient all-reduce under DDP, SyncBatchNorm as the engines wrap it -- by default the host-sync-free
equivalent of unidefense_b200/parallel.py, `--syncbn torch` for the stock class) and the AdamW(amsgrad) update
of the config template.  On one GPU the whole step is captured once and replayed as a CUDA graph (`--graph off`
for eager launches).  Rank 0 prints ONE JSON line (see README / DESIGN.md §5 for the keys).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import torch.nn.functional as F  # noqa: E402

LAMBDAS = dict(triplet=0.1, recons=0.1, freq=1.0, mask=0.1, fac=0.1)   # config_template/forgery/model_udeb4.yml:12-16
ARCH = {"eb4": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2, drop_rate=0.2), 380, 32),
        "r18": ("UDR18", dict(num_classes=2, drop_rate=0.5), 256, 32),
        "r50": ("UDR50", dict(extractor="resnet50", num_classes=2, drop_rate=0.5), 256, 64)}
METRIC = "train samples/sec (fwd+bwd)"


def peaks():
    fn = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(fn):
        return json.load(open(fn)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def synth(n, res, rank, device=None, pin=False):
    g = torch.Generator().manual_seed(1234 + rank)
    x = torch.rand(n, 3, res, res, generator=g) * 2 - 1
    labels = torch.tensor([0] * (n // 2) + [1] * (n - n // 2), dtype=torch.int64)
    if pin:
        x, labels = x.pin_memory(), labels.pin_memory()
    if device is not None:
        x, labels = x.to(device), labels.to(device)
    return x, labels


def init_live(model):
    """SURVEY.md §8(d): make every branch numerically live (sf_coef -10 / fuse_coef 0 would hide the FFT paths)."""
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith("sf_coef"):
                p.fill_(0.0)
            elif n.endswith("fuse_coef"):
                p.fill_(0.3)
            elif p.ndim == 1 and n.endswith("weight"):          # every BN / IN gamma
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
    return model


# ---------------------------------------------------------------------------------------------
# algorithmic bytes per step of each hot-path op (DESIGN.md "kernels"; SURVEY.md §8d formulas)
# ---------------------------------------------------------------------------------------------
def decoder_planes(arch, R):
    """(channels, side) of every InstanceNorm+act plane and the side of the tanh output (SURVEY.md §8a row a2)."""
    if arch == "eb4":
        f = -(-R // 16)            # stride-16 feature, TF-SAME padding: ceil
        return [(80, f), (80, 2 * f), (80, 2 * f), (40, 2 * f), (40, 4 * f), (40, 4 * f), (20, 4 * f), (20, 8 * f),
                (20, 8 * f)], 8 * f
    if arch == "r18":
        f = -(-R // 8)
        return [(128, f), (128, 2 * f), (128, 2 * f), (64, 2 * f), (64, 4 * f), (32, 4 * f)], 4 * f
    f = -(-R // 16)
    return [(256, f), (256, 2 * f), (256, 2 * f), (128, 2 * f), (128, 4 * f), (128, 4 * f), (64, 4 * f), (64, 8 * f),
            (32, 8 * f)], 8 * f


def alg_bytes(arch, N, R, n_real, act_bytes=4):
    """Compulsory HBM bytes per step of each op group: every tensor crossing the group boundary read once + written
    once.  fp32 everywhere except the decoder epilogues, whose activations are `act_bytes` wide (2 under bf16 autocast:
    the bf16 in/out kernels; SURVEY.md §8d "bf16 activations halve G2")."""
    planes, h = decoder_planes(arch, R)
    E = sum(c * s * s for c, s in planes)
    img, dec = 3 * R * R * 4, 3 * h * h * 4
    return {"in_act_fwd": N * 2 * E * act_bytes, "in_act_bwd": N * 3 * E * act_bytes,
            "tanh_fwd": N * 2 * dec, "tanh_bwd": N * 3 * dec,
            "recon_tail_fwd": N * (dec + 2 * img) + 8 * N,
            "recon_tail_bwd": n_real * (dec + img) + N * dec}


# kernel-name pattern -> op group of hot_path.ops_ms_per_step (device time per kernel from CUPTI records)
KERNEL_GROUPS = [("recon_tail_fwd", r"rt2?_(rows_fwd|cols_fwd)_kernel|rt_finalize_kernel"),
                 ("recon_tail_bwd", r"rt2?_(rows_bwd|cols_bwd)_kernel"),
                 ("in_act_fwd", r"ia_fwd"), ("in_act_bwd", r"ia_bwd|ia_param_grad"),
                 ("tanh_fwd", r"ia_tanh_fwd"), ("tanh_bwd", r"ia_tanh_bwd"),
                 ("attn_prep", r"at_prep_kernel"), ("rfft2_cat", r"at_r2c_kernel"), ("irfft2_cat", r"at_c2r_kernel"),
                 ("attn_fuse_fwd", r"at_fuse_fwd"), ("attn_fuse_bwd", r"at_fuse_bwd|at_sum_partials"),
                 ("bn_stats", r"df_bn_stats|pj_merge"), ("dyfi_mask_fwd", r"df_mask_fwd"),
                 ("dyfi_mask_bwd", r"df_mask_bwd|df_w2_reduce"), ("bn_bwd", r"df_bn_bwd"),
                 ("proj_fwd", r"pj_gemm"), ("proj_prep", r"pj_prep"), ("triplet", r"ls_triplet"),
                 ("factorization", r"ls_fac"), ("mask_kl", r"ls_mask_kl|ls_kl_log|ls_sum_kernel"),
                 ("comm_gather", r"cm_gather"), ("sf_pack", r"sf_pack"), ("sf_mix", r"sf_mix|sf_sum"),
                 ("perturb", r"pt_|fs_")]


def cupti_kernel_times(run_step, steps):
    """{group: (launches, total ms)} of OUR kernels over `steps` eager steps, device durations from CUPTI kernel
    records (torch.profiler) -- unlike host-recorded events they do not include launch gaps of a host-bound stream."""
    import re
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            run_step()
        torch.cuda.synchronize()
    out = {}
    pats = [(g, re.compile(p)) for g, p in KERNEL_GROUPS]
    for k in prof.key_averages():
        name = k.key
        t_us = getattr(k, "device_time_total", None)
        if t_us is None:
            t_us = getattr(k, "cuda_time_total", 0.0)
        for g, pat in pats:
            if pat.search(name):
                c, t = out.get(g, (0, 0.0))
                out[g] = (c + k.count, t + t_us / 1e3)
                break
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                    str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([c.strip() for c in o.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "samples": len(sm),
                "power_w_max": max(float(r[2]) for r in self.rows if len(r) > 2), "reasons": reasons}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_arm(arch, res, sample_n, steps, warmup):
    from oracle import ref_model
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    name, kw, _, _ = ARCH[arch]
    torch.manual_seed(0)
    model = init_live(ref_model.build(arch, **kw)).train()
    x, labels = synth(sample_n, res, 0)
    nr = sample_n // 2
    opt = torch.optim.AdamW([p for p in model.parameters() if p.requires_grad], lr=1e-4, weight_decay=5e-6, amsgrad=True)

    def step():
        opt.zero_grad(set_to_none=True)
        out = model(x)
        loss = ref_model.pass1_loss(out, labels, nr, LAMBDAS)
        loss.backward()
        opt.step()
        return float(loss)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return {"value": sample_n / dt, "ms_per_step": dt * 1e3, "cores": threads, "kind": "port",
            "sample": f"{steps} steps of {sample_n} faces at {res}x{res} (fp32, torch CPU, {threads} threads), "
                      f"same model/loss/optimizer"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arch = args.arch
    _, _, res, nb = ARCH[arch]
    res = args.res or res
    r = cpu_arm(arch, res, args.cpu_sample, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"UniDefense {ARCH[arch][0]} train step, {res}x{res}, per-GPU batch {args.batch or nb}",
                       "note": "reference arm = CPU port of the reference (oracle/) on the host cores; bounded sample per step"},
            "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"],
                             "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# isolated recon path: everything downstream of the backbone features, fwd + bwd, on cached features
# ---------------------------------------------------------------------------------------------
RECON_MB_PER_SAMPLE = {("eb4", 380): 71.2, ("r50", 256): 91.0, ("r18", 256): 78.6, ("r18", 380): 176.1}  # SURVEY.md §8(d)


def recon_path_probe(model, arch, nb, res, dev, amp, steps, flush):
    """decoder -> attention -> rec tail -> triplet with the engine's pass-1 weights on random backbone features
    of the config's shapes (BASELINE.md §2 'isolated recon path').  -> ms per fwd+bwd."""
    from unidefense_b200 import ops
    g = torch.Generator().manual_seed(99)
    f16 = -(-res // 16)
    shapes = {"eb4": ((160, f16), (272, -(-res // 32))), "r18": ((448, -(-res // 8)), (512, f16)),
              "r50": ((1024, f16), (2048, -(-res // 32)))}[arch]
    feat = torch.randn(nb, shapes[0][0], shapes[0][1], shapes[0][1], generator=g).to(dev).requires_grad_()
    emb = torch.randn(nb, shapes[1][0], shapes[1][1], shapes[1][1], generator=g).to(dev).requires_grad_()
    x, labels = synth(nb, res, 0, dev)
    r_att = torch.randn(emb.shape, generator=g).to(dev) * 1e-3
    blocks = [getattr(model, f"dec_block{i}") for i in (1, 2, 3) if hasattr(model, f"dec_block{i}")]
    ntri = 2 if arch == "eb4" else 1
    nr = nb // 2
    params = [p for n, p in model.named_parameters() if n.startswith(("dec_block", "freq_filter", "spat_filter", "fuse_coef"))]

    def once():
        for p in params:
            p.grad = None
        feat.grad = emb.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            y, tris = feat, []
            for i, blk in enumerate(blocks):
                if i < ntri:
                    y, t = blk.forward_with_mean(y)
                    tris.append(t)
                else:
                    y = blk(y)
            att = model.attention(y.detach(), x, emb)
        rec, spatial, freq = ops.recon_tail(y.float(), x, model.freq_norm)
        tri = sum(ops.triplet_loss(f, labels) for f in [feat.mean(dim=(-2, -1))] + tris)
        loss = (LAMBDAS["mask"] * att["freq_mask"].mean() + LAMBDAS["mask"] * att["spat_mask"].mean()
                + LAMBDAS["triplet"] * tri + LAMBDAS["recons"] * spatial[:nr].mean() + LAMBDAS["freq"] * freq[:nr].mean()
                + (att["out"] * r_att).sum())
        loss.backward()

    for _ in range(3):
        once()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        once()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / steps


# ---------------------------------------------------------------------------------------------
# the bar: our kernels vs the reference's stock-torch op sequence on the SAME GPU (BASELINE.md §4.5)
# ---------------------------------------------------------------------------------------------
def torch_gpu_bar(arch, nb, res, dev, flush, iters=10):
    """Per op group: ms of our public op vs ms of the torch calls the reference makes (tools/torch_bar.py), same
    tensors, CUDA events, L2 flushed before every iteration.  fwd = forward only, fb = forward + backward."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import torch_bar as TB
    from unidefense_b200 import ops
    planes, h = decoder_planes(arch, res)
    act = "swish" if arch == "eb4" else "relu"
    g = torch.Generator().manual_seed(5)
    out = {}

    def both(name, ours, ref):
        o, _ = TB.time_cuda(ours, iters, flush)
        t, _ = TB.time_cuda(ref, iters, flush)
        out[name] = {"ours_ms": round(o, 4), "torch_ms": round(t, 4), "speedup": round(t / o, 2)}

    dec = torch.tanh(torch.randn(nb, 3, h, h, generator=g)).to(dev).requires_grad_()
    x = (torch.rand(nb, 3, res, res, generator=g) * 2 - 1).to(dev)
    gl = torch.zeros(nb, device=dev)
    gl[: nb // 2] = 1.0 / (nb // 2)

    def tail(fn, bwd):
        def f():
            dec.grad = None
            _, sp, fr = fn(dec, x)
            if bwd:
                torch.autograd.backward([sp, fr], [0.1 * gl, gl])
        return f
    both("recon_tail_fwd", tail(ops.recon_tail, False), tail(TB.recon_tail, False))
    both("recon_tail_fb", tail(ops.recon_tail, True), tail(TB.recon_tail, True))

    xs = [torch.randn(nb, c, s, s, generator=g).to(dev).requires_grad_() for c, s in planes]
    gs = [torch.randn(nb, c, s, s, generator=g).to(dev) for c, s in planes]
    gam = [(torch.rand(c, generator=g) + 0.5).to(dev).requires_grad_() for c, _ in planes]
    bet = [(torch.randn(c, generator=g) * 0.1).to(dev).requires_grad_() for c, _ in planes]

    def inact(fn, bwd):
        def f():
            for xi, gi, ga, be in zip(xs, gs, gam, bet):
                y = fn(xi, ga, be, act)
                if bwd:
                    xi.grad = ga.grad = be.grad = None
                    y.backward(gi)
        return f
    both("in_act_fwd", inact(ops.in_act, False), inact(TB.in_act, False))
    both("in_act_fb", inact(ops.in_act, True), inact(TB.in_act, True))

    C, s = {"eb4": (272, -(-res // 32)), "r18": (512, -(-res // 16)), "r50": (2048, -(-res // 32))}[arch]
    emb = torch.randn(nb, C, s, s, generator=g).to(dev).requires_grad_()
    pred = dec.detach()
    p = TB.attention_params(C, dev)
    r_att = torch.randn(nb, C, s, s, generator=g).to(dev)
    import torch.nn as nn
    from unidefense_b200.model import modules as M
    A = M.MemoryEfficientSwish if act == "swish" else nn.ReLU
    ff = M.FrequencyDynamicFilter(C, A, nn.BatchNorm2d, True, False).to(dev).train()
    sf = M.SpatialDynamicFilter(C, A, nn.BatchNorm2d, True, False).to(dev).train()
    with torch.no_grad():
        ff.layer1[0].weight.copy_(p["fw1"]); ff.layer2[0].weight.copy_(p["fw2"])
        sf.layer1[0].weight.copy_(p["sw1"]); sf.layer2[0].weight.copy_(p["sw2"])
    coef = torch.tensor(0.3, device=dev, requires_grad=True)

    def att_ours():
        emb.grad = None
        sd, fd = ops.attn_prep(pred, x, (s, s), "ortho")
        ef = ops.rfft2_cat(emb, "ortho")
        fo = ff(ef, fd)
        fil = ops.irfft2_cat(fo["out"], (s, s), "ortho")
        sm = sf.mask_only(emb, sd)
        o = ops.attn_fuse(emb, sm, fil, None, coef)
        ((o * r_att).sum() + 0.1 * fo["mask"].mean() + 0.1 * sm.mean()).backward()

    def att_torch():
        emb.grad = None
        o, fm, sm = TB.attention(pred, x, emb, p, act)
        ((o * r_att).sum() + 0.1 * fm.mean() + 0.1 * sm.mean()).backward()
    allow = torch.backends.cudnn.allow_tf32
    both("attention_fb", att_ours, att_torch)
    torch.backends.cudnn.allow_tf32 = allow

    labels = torch.tensor([0] * (nb // 2) + [1] * (nb - nb // 2), device=dev)
    feats = [torch.randn(nb, c, generator=g).to(dev).requires_grad_()
             for c in ((160, 80, 40) if arch == "eb4" else (1024, 256) if arch == "r50" else (448, 128))]

    def tri(fn):
        def f():
            for t in feats:
                t.grad = None
            sum(fn(t, labels) for t in feats).backward()
        return f
    both("triplet_fb", tri(ops.triplet_loss), tri(TB.triplet))

    st = x.flip(0).contiguous()
    lm = (torch.rand(nb, generator=g) / 2 + 0.5).to(dev)
    with torch.no_grad():
        both("freq_style_transfer", lambda: ops.freq_style_transfer(x, st, lm), lambda: TB.freq_style_transfer(x, st, lm))
    return {"what": "our public ops vs the reference's stock-torch op sequence (cuFFT/cuDNN/ATen, fp32) on this GPU; "
                    "fb = forward+backward; CUDA events around the python call, L2 flushed",
            "ops": out, "slower_than_torch": sorted(k for k, v in out.items() if v["speedup"] < 1.0)}


def recon_path_torch_probe(model, arch, nb, res, dev, steps, flush):
    """The isolated recon path (same inputs and loss as recon_path_probe) with every hot-path op issued as the stock
    torch calls of the reference; the decoder / filter convolutions are the same cuDNN calls in both."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import torch_bar as TB
    import torch.nn as nn
    g = torch.Generator().manual_seed(99)
    f16 = -(-res // 16)
    shapes = {"eb4": ((160, f16), (272, -(-res // 32))), "r18": ((448, -(-res // 8)), (512, f16)),
              "r50": ((1024, f16), (2048, -(-res // 32)))}[arch]
    feat = torch.randn(nb, shapes[0][0], shapes[0][1], shapes[0][1], generator=g).to(dev).requires_grad_()
    emb = torch.randn(nb, shapes[1][0], shapes[1][1], shapes[1][1], generator=g).to(dev).requires_grad_()
    x, labels = synth(nb, res, 0, dev)
    r_att = torch.randn(emb.shape, generator=g).to(dev) * 1e-3
    blocks = [getattr(model, f"dec_block{i}") for i in (1, 2, 3) if hasattr(model, f"dec_block{i}")]
    act = "swish" if arch == "eb4" else "relu"
    ntri = 2 if arch == "eb4" else 1
    nr = nb // 2
    fl, sl = model.freq_filter, model.spat_filter
    p = {"fw1": fl.layer1[0].weight, "fg": fl.layer1[1].weight, "fb": fl.layer1[1].bias, "fw2": fl.layer2[0].weight,
         "frm": fl.layer1[1].running_mean.clone(), "frv": fl.layer1[1].running_var.clone(),
         "sw1": sl.layer1[0].weight, "sg": sl.layer1[1].weight, "sb": sl.layer1[1].bias, "sw2": sl.layer2[0].weight,
         "srm": sl.layer1[1].running_mean.clone(), "srv": sl.layer1[1].running_var.clone(), "coef": model.fuse_coef}
    params = [q for n, q in model.named_parameters() if n.startswith(("dec_block", "freq_filter", "spat_filter", "fuse_coef"))]

    def once():
        for q in params:
            q.grad = None
        feat.grad = emb.grad = None
        y, tris = feat, []
        for i, blk in enumerate(blocks):
            mods = list(blk)
            j = 0
            while j < len(mods):
                m = mods[j]
                if isinstance(m, nn.InstanceNorm2d):
                    y = TB.in_act(y, m.weight, m.bias, act)
                    j += 2
                elif isinstance(m, nn.Tanh):
                    y = torch.tanh(y)
                    j += 1
                else:
                    y = m(y)
                    j += 1
            if i < ntri:
                tris.append(y.mean(dim=(-2, -1)))
        out, fm, sm = TB.attention(y.detach(), x, emb, p, act, model.freq_norm)
        rec, spatial, freq = TB.recon_tail(y, x, model.freq_norm)
        tri = sum(TB.triplet(f, labels) for f in [feat.mean(dim=(-2, -1))] + tris)
        loss = (LAMBDAS["mask"] * fm.mean() + LAMBDAS["mask"] * sm.mean() + LAMBDAS["triplet"] * tri
                + LAMBDAS["recons"] * spatial[:nr].mean() + LAMBDAS["freq"] * freq[:nr].mean() + (out * r_att).sum())
        loss.backward()

    for _ in range(3):
        once()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        once()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / steps


# ---------------------------------------------------------------------------------------------
# C5 (BASELINE.json configs[4]): frequency-branch microbench sweep
# ---------------------------------------------------------------------------------------------
def run_microbench(args):
    """R in {224, 299, 380} x B in {16..256}: the fused reconstruction loss (upsample + FFT2 + spectral/spatial L1),
    forward and forward+backward, and FrequencyStyleTransfer (FFT2 x2 + amplitude mix + IFFT2), ours vs the stock
    torch sequence; algorithmic bytes per SURVEY.md §8(d)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import torch_bar as TB
    from unidefense_b200 import ops
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    pk, pk_kind = peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rows = []
    for R in (224, 299, 380):
        h = R // 2 + (R % 2) if R != 380 else 192          # the decoder reconstructs at ~half resolution
        for B in (16, 32, 64, 128, 256):
            g = torch.Generator().manual_seed(R + B)
            x = (torch.rand(B, 3, R, R, generator=g) * 2 - 1).to(dev)
            dec = torch.tanh(torch.randn(B, 3, h, h, generator=g)).to(dev).requires_grad_()
            gl = torch.full((B,), 1.0 / B, device=dev)
            img, dch = 3 * R * R * 4, 3 * h * h * 4
            it = max(3, min(args.steps, 10))

            def tail(fn, bwd):
                def f():
                    dec.grad = None
                    _, sp, fr = fn(dec, x)
                    if bwd:
                        torch.autograd.backward([sp, fr], [0.1 * gl, gl])
                return f
            st = x.flip(0).contiguous()
            lm = (torch.rand(B, generator=g) / 2 + 0.5).to(dev)
            cases = [("recon_loss_fwd", tail(ops.recon_tail, False), tail(TB.recon_tail, False), B * (dch + 2 * img)),
                     ("recon_loss_fwd_bwd", tail(ops.recon_tail, True), tail(TB.recon_tail, True),
                      B * (dch + 2 * img) + B * (2 * dch + img)),
                     ("freq_style_transfer", lambda: ops.freq_style_transfer(x, st, lm),
                      lambda: TB.freq_style_transfer(x, st, lm), B * 3 * img)]
            # the composite BASELINE.json names: FFT2 + spectral mask + IFFT2 + L1 loss against a target (SURVEY §8d:
            # read x + read half-spectrum mask + write y + read target), and the rank-matching perturbation (a14)
            mk = torch.rand(B, R, R // 2 + 1, generator=g).to(dev)

            def comp_ours():
                return (ops.spectral_mask_filter(x, mk) - st).abs().mean(dim=(1, 2, 3))

            def comp_torch():
                f = torch.fft.rfft2(x, norm="ortho") * mk.unsqueeze(1)
                return (torch.fft.irfft2(f, s=(R, R), norm="ortho") - st).abs().mean(dim=(1, 2, 3))

            def sst_torch():
                cf, sf_ = x.flatten(2), st.flatten(2)
                idx = torch.sort(cf, dim=-1).indices
                vs = torch.sort(sf_, dim=-1).values
                l3 = lm.view(-1, 1, 1)
                return (cf + (1 - l3) * vs.gather(-1, idx.argsort(-1)) - (1 - l3) * cf).view_as(x)
            if B <= 64:                      # (the sort workspace is 5 x the batch; the stock path 4 sorts of it)
                cases += [("fft2_mask_ifft2_l1", comp_ours, comp_torch, B * (3 * img + 3 * R * (R // 2 + 1) * 4)),
                          ("spatial_style_transfer", lambda: ops.spatial_style_transfer(x, st, lm), sst_torch, B * 3 * img)]
            for name, ours, ref, nbytes in cases:
                with torch.set_grad_enabled(name in ("recon_loss_fwd", "recon_loss_fwd_bwd")):
                    o, ob = TB.time_cuda(ours, it, flush)
                    t, _ = TB.time_cuda(ref, it, flush)
                gbs = nbytes / (o * 1e-3) / 1e9
                rows.append({"op": name, "R": R, "B": B, "ours_ms": round(o, 4), "ours_best_ms": round(ob, 4),
                             "torch_ms": round(t, 4), "speedup": round(t / o, 2), "alg_mb": round(nbytes / 1e6, 2),
                             "gbs": round(gbs, 1), "hbm_frac": round(gbs / pk["hbm_gbs"], 4)})
            del x, dec, st
            torch.cuda.empty_cache()
    print(json.dumps({"microbench": "C5 frequency-branch sweep (BASELINE.json configs[4])", "peak_hbm_gbs": pk["hbm_gbs"],
                      "peak_kind": pk_kind, "unit": "ms per call, CUDA events, L2 flushed", "rows": rows}), flush=True)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
DUMP_LIMIT = 64 * 10 ** 6          # bytes of all files written by --dump-outputs together


def dump_outputs(outdir, last, params):
    """Writes what the last timed step computed as <outdir>/<name>.npy (float32; float64 stays float64): the loss, every
    tensor of the model's output dict (`cls_out`, `rec`, `loss_dict.<key>`, `loss_dict.triplet.<i>`), and the gradients
    and updated values of the trained parameters, each flattened and concatenated in model.parameters() order.  An
    array larger than its equal share of DUMP_LIMIT is replaced by the same seeded sample of its flattened elements
    (sorted indices) on every run, so two builds run with the same arguments can be compared file by file.  Inputs and
    initial weights are seeded and the step is deterministic (see run_ours), so two runs of one build write the same
    files."""
    import numpy as np
    arrays = {"loss": last["loss"]}

    def add(name, v):
        if torch.is_tensor(v):
            arrays[name] = v
        elif isinstance(v, dict):
            for k, x in v.items():
                add(f"{name}.{k}" if name else k, x)
        elif isinstance(v, (list, tuple)):
            for i, x in enumerate(v):
                add(f"{name}.{i}", x)
    add("", last["out"])
    arrays["param_grads"] = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).flatten() for p in params])
    arrays["params"] = torch.cat([p.detach().flatten() for p in params])
    os.makedirs(outdir, exist_ok=True)
    share = DUMP_LIMIT // len(arrays) - 4096                  # (room for the .npy header)
    for name, t in arrays.items():
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 else t.float()
        keep = share // t.element_size()
        if t.numel() > keep:
            idx = torch.randint(t.numel(), (keep,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.flatten()[idx.to(t.device)]
        np.save(os.path.join(outdir, f"{name}.npy"), t.cpu().numpy())


def run_ours(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    flat_dp = world > 1 and args.dp == "flat"
    ddp_graph = world > 1 and (flat_dp or args.graph == "on" or os.environ.get("UD_BENCH_DDP_GRAPH", "0") == "1")
    if args.graph == "off":
        ddp_graph = False
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from unidefense_b200 import _lib as L
    from unidefense_b200 import ops
    from unidefense_b200.model import load_model

    arch = args.arch
    name, kw, res, nb = ARCH[arch]
    res, nb = args.res or res, args.batch or nb
    torch.manual_seed(0)
    # Same arguments, same result: the reference engines time cuDNN's algorithms per process (cudnn.benchmark,
    # engine/abstract_engine.py:120), which picks differently from run to run, and some of those algorithms add with
    # atomics; either makes two runs of one build train to different weights.  Deterministic algorithms, chosen by
    # cuDNN's heuristics, make the step bit-reproducible (our kernels reduce in a fixed order).
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.deterministic = True
    model = init_live(load_model(name)(**kw)).to(dev).train()
    if args.channels_last == "all":
        model = model.to(memory_format=torch.channels_last)
    elif args.channels_last == "backbone":          # stock-torch part only; the hot path's convs stay NCHW like its kernels
        for part in ("backbone", "extractor", "emb_block1", "emb_block2"):
            if hasattr(model, part):
                getattr(model, part).to(memory_format=torch.channels_last)
    if world > 1:                                             # engine/forgery_engine.py:142-145
        if args.syncbn == "torch":
            model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)
        else:       # same math and collectives, without torch's per-layer device->host sync (unidefense_b200/parallel.py)
            from unidefense_b200.parallel import convert_sync_batchnorm
            model = convert_sync_batchnorm(model)
        if flat_dp:
            # B200-native data parallelism (unidefense_b200/parallel.py): SyncBatchNorm statistics over NVLink peer
            # memory (one single-CTA kernel per exchange, csrc/ud_comm.cu) and ONE NCCL all-reduce of a flat gradient
            # buffer -- no DDP reducer, so the whole step (collectives included) replays as one CUDA graph
            from unidefense_b200.parallel import FlatGradients, PeerComm, set_default_comm
            comm = PeerComm(max_count=16384)
            set_default_comm(comm)
            ddp = model
            flat = FlatGradients(model.parameters())
        else:
            ctor_stream = torch.cuda.Stream() if ddp_graph else torch.cuda.current_stream()
            with torch.cuda.stream(ctor_stream):       # DDP must be built on a side stream to be capturable later
                ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=False)
            torch.cuda.current_stream().wait_stream(ctor_stream)
            flat = None
    else:
        ddp = model
        flat = None
    params = [p for p in model.parameters() if p.requires_grad]
    # whole-step CUDA graph: validated single-GPU; under DDP the NCCL capture dead-locked on this stack (round 1),
    # so multi-GPU runs stay eager unless --graph on is forced
    use_graph = (args.graph != "off" and world == 1) or ddp_graph
    opt = torch.optim.AdamW(params, lr=1e-4, betas=(0.9, 0.999), weight_decay=5e-6, amsgrad=True, fused=True,
                            capturable=use_graph)
    x_host, l_host = synth(nb, res, rank, pin=True)
    x_dev, l_dev = x_host.to(dev), l_host.to(dev)
    nr = nb // 2
    amp = args.dtype == "bf16"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    # --dump-outputs: loss and model outputs of the one step recorded (the capture, whose static outputs every replay
    # rewrites, or the last timed eager step); no other step keeps its outputs alive, so memory use matches a plain run
    last = {"record": False}

    def body(x, labels):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            out = ddp(x)
        ld = out["loss_dict"]
        tri = sum(ops.triplet_loss(f, labels) for f in ld["triplet"])
        loss = (ops.cross_entropy(out["cls_out"].float(), labels) + LAMBDAS["mask"] * ld["freq_mask"].mean()
                + LAMBDAS["mask"] * ld["spat_mask"].mean() + LAMBDAS["triplet"] * tri
                + LAMBDAS["recons"] * ld["spatial"][:nr].mean() + LAMBDAS["freq"] * ld["freq"][:nr].mean())
        loss.backward()
        if flat is not None:
            flat.all_reduce()                       # one NCCL all-reduce (avg) of every gradient
        opt.step()
        if last["record"]:
            last.update(loss=loss, out=out)
        return loss

    def second_pass(x, labels, gt):
        """engine/abstract_engine.py:286-376: perturbed forward (host-RNG augmentation dispatch incl. coral / style
        transfer / noise / blur / downscale), KL mask alignment against pass 1 (steady state: cur_step > 10 %),
        factorization loss against pass 1, 0.1-weighted CE / rec / freq, backward, optimizer step."""
        perm_r = torch.arange(nr)[torch.randperm(nr)]
        perm_f = torch.arange(nb - nr)[torch.randperm(nb - nr)]
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            out = ddp(x, pert_real_list=perm_r, pert_fake_list=perm_f, preserve_color=True)
        ld = out["loss_dict"]
        tri = sum(ops.triplet_loss(f, labels) for f in ld["triplet"])
        fm = ops.mask_kl_loss(ld["freq_mask"], gt["freq_mask"])
        sm = ops.mask_kl_loss(ld["spat_mask"], gt["spat_mask"])
        fac = ops.factorization_loss(ld["factorization"].float(), gt["fac"])
        loss = (0.1 * ops.cross_entropy(out["cls_out"].float(), labels) + LAMBDAS["mask"] * fm + LAMBDAS["mask"] * sm
                + LAMBDAS["triplet"] * tri + LAMBDAS["recons"] * 0.1 * ld["spatial"][:nr].mean()
                + LAMBDAS["freq"] * 0.1 * ld["freq"][:nr].mean() + LAMBDAS["fac"] * fac)
        loss.backward()
        if flat is not None:
            flat.all_reduce()
        opt.step()
        if last["record"]:
            last.update(loss=loss, out=out)
        return loss

    def two_pass_step(x, labels):
        """One engine iteration = clean pass + perturbed pass (engine/abstract_engine.py:207-381), eager."""
        zero_grads()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            out = ddp(x)
        ld = out["loss_dict"]
        gt = {"freq_mask": ld["freq_mask"].detach().clone(), "spat_mask": ld["spat_mask"].detach().clone(),
              "fac": ld["factorization"].detach().float().clone()}
        tri = sum(ops.triplet_loss(f, labels) for f in ld["triplet"])
        loss = (ops.cross_entropy(out["cls_out"].float(), labels) + LAMBDAS["mask"] * ld["freq_mask"].mean()
                + LAMBDAS["mask"] * ld["spat_mask"].mean() + LAMBDAS["triplet"] * tri
                + LAMBDAS["recons"] * ld["spatial"][:nr].mean() + LAMBDAS["freq"] * ld["freq"][:nr].mean())
        loss.backward()
        if flat is not None:
            flat.all_reduce()
        opt.step()
        zero_grads()
        return second_pass(x, labels, gt)

    def zero_grads():
        if flat is not None:
            flat.zero()                             # gradients are views into the flat buffer: keep them
        else:
            opt.zero_grad(set_to_none=True)

    def eager_step(x, labels):
        zero_grads()
        return body(x, labels)

    step = two_pass_step if args.two_pass else eager_step
    if args.two_pass:
        use_graph = False                      # the augmentation dispatch draws from the host RNG every iteration
    graph_note = "off" if world == 1 or args.graph == "off" else "off (eager under DDP: NCCL capture not validated)"
    graph_launches = 0
    if args.two_pass:
        graph_note = "off (two-pass engine iteration: host-RNG augmentation dispatch)"
    if use_graph:
        # Whole-step CUDA graph (forward, loss, backward incl. DDP/SyncBN NCCL collectives, fused AdamW): the step
        # issues ~3000 small kernels and is host-launch-bound, worst with 8 ranks sharing the box's cores.
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(11 if (world > 1 and flat is None) else 3):   # DDP needs 11 side-stream iterations before capture
                    eager_step(x_dev, l_dev)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            if flat is None:
                opt.zero_grad(set_to_none=True)
            l0 = L.lib().ud_launch_count()
            err = None
            last["record"] = bool(args.dump_outputs)
            try:
                with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                    if flat is not None:
                        flat.zero()
                    static_loss = body(x_dev, l_dev)
            except Exception as e:                   # noqa: BLE001
                err = e
            last["record"] = False
            graph_launches = L.lib().ud_launch_count() - l0
            if world > 1:                            # every rank replays, or none does (else the collectives dead-lock)
                flag = torch.tensor([0.0 if err is not None else 1.0], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                if float(flag) == 0.0 and err is None:
                    err = RuntimeError("capture failed on another rank")
            if err is not None:
                raise err
            graph.replay()
            torch.cuda.synchronize()
            if not bool(torch.isfinite(static_loss)):
                raise RuntimeError("non-finite loss after graph replay")

            def step(x, labels):
                if x is not x_dev:
                    x_dev.copy_(x, non_blocking=True)
                    l_dev.copy_(labels, non_blocking=True)
                graph.replay()
                return static_loss
            graph_note = "whole step captured"
        except Exception as e:                       # fall back to eager launches, say so in the JSON line
            if args.graph == "on" and world == 1:
                raise
            graph_note = f"capture failed, eager ({type(e).__name__}: {str(e)[:120]})"
            torch.cuda.synchronize()
            step = eager_step
            use_graph = False

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.recon_only:
        ms_ = recon_path_probe(model, arch, nb, res, dev, amp, args.steps, flush)
        print(json.dumps({"recon_only_ms": ms_, "samples_per_s": nb / (ms_ * 1e-3)}), flush=True)
        return
    for _ in range(args.warmup):
        step(x_dev, l_dev)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None     # one nvidia-smi poller per job, not per rank
    if sampler is not None:
        sampler.start()
    graphed = graph_note == "whole step captured"
    launches0 = L.lib().ud_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        flush.zero_()                                          # L2 flush between timed iterations
        if args.dump_outputs and not graphed and i == args.steps - 1:
            last["record"] = True
        step(x_dev, l_dev)
    e1.record()
    last["record"] = False
    barrier()
    launches = graph_launches * args.steps if graphed else L.lib().ud_launch_count() - launches0
    ms = e0.elapsed_time(e1) / args.steps
    clocks = sampler.summary() if sampler is not None else None
    if args.dump_outputs and rank == 0:          # before the steps below move the weights on
        dump_outputs(args.dump_outputs, last, params)
    # per-op device times behind `roofline` / `hot_path`: the same step issued eagerly right after the timed region
    # (same inputs, same kernels, L2 flushed), kernel durations taken from CUPTI records; host-recorded events (the
    # round-1 method) are only the fallback because in a host-bound eager stream they include the launch gaps
    L.PROFILE = None
    prof_steps = min(args.steps, 3)

    def _prof_step():
        flush.zero_()
        eager_step(x_dev, l_dev)
    try:
        if rank == 0:
            prof = cupti_kernel_times(_prof_step, prof_steps)
        else:                                # the other ranks only keep the collectives of those steps company
            prof = {}
            for _ in range(prof_steps):
                _prof_step()
            torch.cuda.synchronize()
        prof_how = "CUPTI kernel records (torch.profiler) of the step re-issued eagerly after the timed region"
    except Exception as e:                   # noqa: BLE001
        prof = {}
        if world == 1:                       # (at N>1 extra steps on one rank would unbalance the collectives)
            L.PROFILE = {}
            for _ in range(prof_steps):
                _prof_step()
            torch.cuda.synchronize()
            prof = L.profile_summary()
            L.PROFILE = None
        prof_how = f"CUDA events around each C-ABI call (CUPTI unavailable: {type(e).__name__})"

    # end to end through the public API with HOST buffers: pinned H2D of the batch + D2H of the loss every step
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        if graphed:
            loss = step(x_host, l_host)                      # H2D straight into the graph's static input buffers
        else:
            loss = step(x_host.to(dev, non_blocking=True), l_host.to(dev, non_blocking=True))
        loss_host = loss.item()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    t = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])

    recon_ms = recon_torch_ms = bar = None
    if world == 1 and not args.no_recon_probe:
        L.PROFILE = {}
        recon_ms = recon_path_probe(model, arch, nb, res, dev, amp, max(args.steps, 5), flush)
        recon_prof = {k: v[1] / max(args.steps, 5) for k, v in L.profile_summary().items()}
        L.PROFILE = None
        recon_f32_ms = recon_path_probe(model, arch, nb, res, dev, False, max(args.steps, 5), flush)
        recon_torch_ms = recon_path_torch_probe(model, arch, nb, res, dev, max(args.steps, 5), flush)
        bar = torch_gpu_bar(arch, nb, res, dev, flush)

    if rank == 0:
        pk, pk_kind = peaks()
        act_bytes = 2 if args.dtype == "bf16" else 4
        ab = alg_bytes(arch, nb, res, nr, act_bytes)
        ops_ms = {k: v[1] / prof_steps for k, v in prof.items()}
        timed = {k: (ab[k] / (ops_ms[k] * 1e-3) / 1e9) for k in ab if k in ops_ms and ops_ms[k] > 0}
        dom = max((k for k in ops_ms if k in ab), key=lambda k: ops_ms[k], default=None)
        roof = None
        if dom:
            ach = timed[dom]
            roof = {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": pk["hbm_gbs"], "peak_kind": pk_kind,
                    "unit": "GB/s", "frac": round(ach / pk["hbm_gbs"], 4), "traffic": TRAFFIC.get(dom),
                    "alg_bytes_per_launch": ab[dom] // max(prof[dom][0] // prof_steps, 1),
                    "launches_per_step": prof[dom][0] // prof_steps, "timed_with": prof_how,
                    "ms_per_step_in_kernel": round(ops_ms[dom], 4)}
        sf_ms = sum(v for k, v in ops_ms.items() if k.startswith("sf_"))     # SFConv glue (backbone, §8f) -- not recon path
        dense_ms = ops_ms.get("proj_fwd", 0.0) + ops_ms.get("proj_prep", 0.0)   # tcgen05 projections: tensor-pipe bound
        comm_ms = ops_ms.get("comm_gather", 0.0)
        hot_ms = sum(ops_ms.values()) - sf_ms - dense_ms - comm_ms
        mbs = RECON_MB_PER_SAMPLE.get((arch, res))
        if mbs and act_bytes == 2:               # SURVEY's figure counts fp32 epilogue activations: take half of G2 off
            f32 = alg_bytes(arch, 1, res, 1, 4)
            mbs = round(mbs - 0.5 * (f32["in_act_fwd"] + f32["in_act_bwd"]) / 1e6, 2)
        line = {"metric": METRIC, "value": round(nb * world / (ms * 1e-3), 2), "unit": "samples/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": (f"UniDefense {name} two-pass engine iteration (clean pass + perturbed pass with "
                                        f"KL mask alignment and factorization loss, 2 x (fwd + bwd + AdamW amsgrad)), "
                                        if args.two_pass else
                                        f"UniDefense {name} train step (fwd + engine pass-1 loss + bwd + AdamW amsgrad), ")
                                       + f"{res}x{res}, per-GPU batch {nb}, random init",
                           "hot_path_dtype": "f32" if act_bytes == 4 else
                                             "f32 arithmetic; decoder epilogues bf16 in / bf16 out (algorithmic bytes counted at 2 B)",
                           "backbone": f"stock torch, {args.dtype} autocast"
                                       + (f", channels_last ({args.channels_last})" if args.channels_last != "none" else ""),
                           "parallelism": f"dp{world}" + ((" (flat-gradient NCCL all-reduce + SyncBatchNorm over NVLink peer memory)"
                                                            if flat is not None else
                                                            f" (DDP + SyncBatchNorm[{args.syncbn}], NCCL)") if world > 1 else ""),
                           "cuda_graph": graph_note,
                           "l2": "256 MB buffer written between timed iterations; per-step activations >> 126 MB L2"},
                "clocks": clocks,
                "e2e": {"value": round(nb * world / (e2e_ms * 1e-3), 2), "unit": "samples/s",
                        "h2d_bytes_per_step": x_host.numel() * 4 + l_host.numel() * 8, "d2h_bytes_per_step": 4,
                        "ms_per_step": round(e2e_ms, 3), "last_loss": loss_host},
                "gpu_launches": int(launches),
                "roofline": roof,
                "hot_path": {"kernel_ms_per_step": round(hot_ms, 3), "share_of_step": round(hot_ms / ms, 4),
                             "sfconv_glue_kernel_ms_per_step": round(sf_ms, 3),
                             "tcgen05_projection_ms_per_step": round(dense_ms, 3),
                             "peer_exchange_ms_per_step": round(comm_ms, 3),
                             "alg_mb_per_sample": mbs,
                             "hbm_frac_of_recon_path_kernels": (round(mbs * 1e6 * nb / (hot_ms * 1e-3) / 1e9 / pk["hbm_gbs"], 4)
                                                                if mbs and hot_ms > 0 else None),
                             "ops_ms_per_step": {k: round(v, 4) for k, v in sorted(ops_ms.items(), key=lambda kv: -kv[1])},
                             "ops_gbs": {k: round(v, 1) for k, v in timed.items()}}}
        if recon_ms is not None:
            mb = mbs                                 # (bf16-adjusted like hot_path.alg_mb_per_sample)
            kern_ms = sum(recon_prof.values())
            line["recon_path"] = {
                "what": "isolated recon path fwd+bwd on cached backbone features (decoder incl. cuDNN convs, attention, "
                        "rec tail, triplet)", "ms": round(recon_ms, 3), "samples_per_s": round(nb / (recon_ms * 1e-3), 1),
                "alg_mb_per_sample": mb,
                "hbm_frac_whole_path": round(mb * 1e6 * nb / (recon_ms * 1e-3) / 1e9 / pk["hbm_gbs"], 4) if mb else None,
                "ms_fp32": round(recon_f32_ms, 3), "torch_gpu_ms": round(recon_torch_ms, 3),
                "speedup_vs_torch_gpu": round(recon_torch_ms / recon_f32_ms, 2),
                "note": "includes the library convolutions (dense, not in the algorithmic bytes) and host launch gaps; "
                        "the kernels-only fraction is hot_path.hbm_frac_of_recon_path_kernels, timed inside the step. "
                        "ms = bench configuration (bf16 autocast convs); ms_fp32 / torch_gpu_ms = everything fp32: ours "
                        "vs the reference's stock-torch op sequence (cuFFT/cuDNN/ATen) on this GPU"}
            line["torch_gpu_bar"] = bar
            del kern_ms
        if world == 1 and not args.no_cpu_baseline:
            c = cpu_arm(arch, res, args.cpu_sample, 2, 1)
            line["cpu_baseline"] = {"value": round(c["value"], 3), "unit": "samples/s", "cores": c["cores"],
                                    "kind": c["kind"], "sample": c["sample"]}
        print(json.dumps(line), flush=True)
    if world > 1:
        # every rank is done with collectives (the MAX all-reduce above was the last one).  Tearing the process group
        # down after NCCL work has been captured into a CUDA graph was observed to hang at 8 ranks until the launcher's
        # timeout; the line is printed, so leave without the graceful teardown.
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize()
        os._exit(0)


# DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, averaged over the launches of the group in one
# step) from the committed ncu pass over the same kernels at the same shapes: profiles/r02_traffic.json, written by
# tools/ncu_traffic.py.  None for a group that has not been captured.
def _load_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            return {k: v["dram_bytes_per_launch"] for k, v in json.load(f)["groups"].items()}
    except (OSError, ValueError, KeyError):
        return {}


TRAFFIC = _load_traffic()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--arch", default="eb4", choices=list(ARCH))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the config's)")
    ap.add_argument("--res", type=int, default=0)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--channels-last", default="backbone", choices=["none", "all", "backbone"],
                    help="memory format of the stock-torch convolutions (the hot-path kernels are NCHW)")
    ap.add_argument("--cpu-sample", type=int, default=4, help="faces per CPU step of the reference / cpu_baseline leg")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="capture the whole training step in a CUDA graph (auto: fall back to eager if capture fails)")
    ap.add_argument("--dp", default="flat", choices=["flat", "ddp"],
                    help="multi-GPU plumbing: flat = one flat-gradient all-reduce + peer-memory SyncBN statistics "
                         "(CUDA-graph replay); ddp = torch DistributedDataParallel as the reference engines wrap it")
    ap.add_argument("--syncbn", default="ours", choices=["ours", "torch"],
                    help="multi-GPU BatchNorm conversion: torch.nn.SyncBatchNorm or the host-sync-free equivalent")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-recon-probe", action="store_true")
    ap.add_argument("--recon-only", action="store_true", help="run only the isolated recon-path probe (profiling aid)")
    ap.add_argument("--two-pass", action="store_true",
                    help="time the reference's full engine iteration (clean + perturbed pass, config C4) instead of one pass")
    ap.add_argument("--microbench", action="store_true",
                    help="C5 (BASELINE.json configs[4]): frequency-branch sweep R in {224,299,380} x B in {16..256}")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write what the last one computed to DIR/<name>.npy (seeded inputs: "
                         "runs with the same arguments compare output for output; at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.microbench or args.recon_only):
        ap.error("--dump-outputs applies to the timed training step of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.microbench:
        run_microbench(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
