import os, sys, torch, torch.nn.functional as F
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import procedural as P
F.dropout = lambda t, p=0.5, training=True, inplace=False: t * 1.0
torch.backends.cudnn.deterministic = True
from unidefense_b200.model import load_model, sfconv
from unidefense_b200 import ops
dft_gemm_ok = sfconv._dft_gemm_ok

def build(arch):
    name, kw = {"eb4": ("UDEB4", dict(extractor="efficientnet-b4", num_classes=2, drop_rate=0.0, drop_connect_rate=0.0)),
                "r18": ("UDR18", dict(num_classes=2, drop_rate=0.0))}[arch]
    m = load_model(name)(**kw)
    P.fill_state_dict_(m, prefix_filter=None, salt=5)
    return m.cuda().train()

def rel2(a, b):
    a, b = a.detach().float().flatten(), b.detach().float().flatten()
    return float((a - b).norm() / b.norm())

for arch in ("eb4", "r18"):
    n, res = 16, 128
    g = torch.Generator().manual_seed(77)
    x = (torch.rand(n, 3, res, res, generator=g) * 2 - 1).cuda()
    torch.backends.cudnn.allow_tf32 = False
    ref = build(arch)(x)
    for tag, dft, cl, tf32 in (("bench config", True, True, True), ("DFT-GEMM off (cuFFT fp32)", False, True, True),
                               ("DFT-GEMM off, NCHW", False, False, True), ("bench config, 3xTF32 projections", True, True, False)):
        sfconv._dft_gemm_ok = dft_gemm_ok if dft else (lambda x: False)      # "DFT-GEMM off": the cuFFT glue path
        m = build(arch)
        if cl:
            for part in ("backbone", "extractor", "emb_block1", "emb_block2"):
                if hasattr(m, part):
                    getattr(m, part).to(memory_format=torch.channels_last)
        torch.backends.cudnn.allow_tf32 = tf32
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = m(x)
        torch.backends.cudnn.allow_tf32 = False
        a, b = out["loss_dict"], ref["loss_dict"]
        print(f"{arch} {tag:36s} rec {rel2(out['rec'], ref['rec']):.3f} cls {rel2(out['cls_out'], ref['cls_out']):.3f} "
              f"fmask {rel2(a['freq_mask'], b['freq_mask']):.3f} smask {rel2(a['spat_mask'], b['spat_mask']):.3f} "
              f"tri0 {rel2(a['triplet'][0], b['triplet'][0]):.3f} fac {rel2(a['factorization'], b['factorization']):.3f} "
              f"spatial {rel2(a['spatial'], b['spatial']):.4f}", flush=True)
    sfconv._dft_gemm_ok = dft_gemm_ok
