"""torch.autograd.Function wrappers over the C ABI (one per hot-path row of SURVEY.md §8a)."""
import torch

from . import _lib as L


def norm_flag(norm):
    """torch.fft `norm` argument -> the kernels' flag.  The reference forwards freq_norm verbatim to torch.fft
    (model/unidefense.py:130-145,:246-249); 'forward' scaling is not on any shipped config and is rejected loudly
    rather than silently computed as 'backward'."""
    if norm in (None, "backward"):
        return 0
    if norm == "ortho":
        return 1
    raise ValueError(f"freq_norm={norm!r} is not supported by the sm_100a kernels (None / 'backward' / 'ortho')")


class _ReconTail(torch.autograd.Function):
    """a1: model/unidefense.py:244-253 / :423-433 / :618-628.  Differentiable in dec and in x (rec - x and rfft2(x) are
    differentiated in the reference); the x gradient is only computed when x requires one."""

    @staticmethod
    def forward(ctx, dec, x, norm_ortho):
        dec = dec.contiguous()
        x = x.contiguous()
        L.require_cuda_f32(dec, x)
        N, C, h, w = dec.shape
        H, W = x.shape[-2:]
        if x.shape[0] != N or x.shape[1] != C:
            raise ValueError(f"recon_tail: dec {tuple(dec.shape)} and x {tuple(x.shape)} disagree")
        lib = L.lib()
        rec = torch.empty_like(x)
        spatial = torch.empty(N, device=x.device, dtype=torch.float32)
        freq = torch.empty(N, device=x.device, dtype=torch.float32)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        signs = (torch.empty(lib.ud_recon_tail_signs_bytes(N, C, H, W), dtype=torch.uint8, device=x.device)
                 if need_grad else None)
        nws = lib.ud_recon_tail_workspace_bytes(N, C, h, w, H, W)
        ws = L.workspace(nws, x.device)
        L.check(lib.ud_recon_tail_fwd(L.ptr(dec), L.ptr(x), L.ptr(rec), L.ptr(spatial), L.ptr(freq), L.ptr(signs),
                                      L.ptr(ws), ws.numel(), N, C, h, w, H, W, int(norm_ortho), L.stream()),
                "recon_tail_fwd")
        if need_grad:
            ctx.save_for_backward(dec, x, signs)
        ctx.norm_ortho = int(norm_ortho)
        ctx.set_materialize_grads(False)          # unused outputs (rec, in training) arrive as None, not as zeros
        return rec, spatial, freq

    @staticmethod
    def backward(ctx, g_rec, g_spatial, g_freq):
        dec, x, signs = ctx.saved_tensors
        N, C, h, w = dec.shape
        H, W = x.shape[-2:]
        lib = L.lib()
        need_dec, need_x = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        g_dec = g_x = None
        if g_spatial is not None or g_freq is not None:
            gs = (g_spatial if g_spatial is not None else torch.zeros(N, device=x.device)).contiguous().float()
            gf = (g_freq if g_freq is not None else torch.zeros(N, device=x.device)).contiguous().float()
            g_dec = torch.empty_like(dec) if need_dec else None
            g_x = torch.empty_like(x) if need_x else None
            nws = lib.ud_recon_tail_workspace_bytes(N, C, h, w, H, W)
            ws = L.workspace(nws, x.device)
            L.check(lib.ud_recon_tail_bwd(L.ptr(dec), L.ptr(x), L.ptr(signs), L.ptr(gs), L.ptr(gf), L.ptr(g_dec),
                                          L.ptr(g_x), L.ptr(ws), ws.numel(), N, C, h, w, H, W, ctx.norm_ortho, L.stream()),
                    "recon_tail_bwd")
        if g_rec is not None and need_dec:
            # rec = interpolate(dec) is differentiable in the reference (model/unidefense.py:244); the shipped engines
            # never use that gradient, but a loss on out['rec'] gets the transposed resize, not silent zeros
            g_up = torch.empty_like(dec)
            L.check(lib.ud_bilinear_ac_bwd(L.ptr(g_rec.contiguous().float()), L.ptr(g_up), N * C, h, w, H, W, L.stream()),
                    "bilinear_bwd")
            g_dec = g_up if g_dec is None else g_dec + g_up
        return g_dec, g_x, None


def recon_tail(dec, x, norm="ortho"):
    """-> (rec [N,C,H,W], spatial [N], freq [N]); rec is differentiable w.r.t. dec, spatial and freq w.r.t. dec and x."""
    return _ReconTail.apply(dec, x, norm_flag(norm))


ACT_CODES = {"none": 0, "relu": 1, "swish": 2}


class _InAct(torch.autograd.Function):
    """a2: InstanceNorm2d(affine) + Swish/ReLU in one pass (model/unidefense.py:61-98 etc.).  x may be fp32 or bf16
    (the output, the saved input and the input gradient keep x's dtype; statistics, parameters and ymean are fp32)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, act, eps, want_mean):
        x = x.contiguous()
        L.require_cuda_f32(x, also=(torch.bfloat16,))
        L.require_cuda_f32(gamma, beta)
        N, C = x.shape[:2]
        HW = x[0, 0].numel() if N > 0 else int(torch.tensor(x.shape[2:]).prod())
        lib = L.lib()
        y = torch.empty_like(x)
        mean = torch.empty(N * C, device=x.device, dtype=torch.float32)
        rstd = torch.empty(N * C, device=x.device, dtype=torch.float32)
        ymean = torch.empty(N, C, device=x.device, dtype=torch.float32) if want_mean else None
        fwd = lib.ud_in_act_fwd_bf16 if x.dtype == torch.bfloat16 else lib.ud_in_act_fwd
        L.check(fwd(L.ptr(x), L.ptr(gamma), L.ptr(beta), L.ptr(y), L.ptr(mean), L.ptr(rstd), L.ptr(ymean), N, C, HW,
                    float(eps), act, L.stream()), "in_act_fwd")
        ctx.save_for_backward(x, gamma, beta, mean, rstd)
        ctx.act = act
        ctx.hw = HW
        if want_mean:
            return y, ymean
        return y, None

    @staticmethod
    def backward(ctx, gy, g_ymean):
        x, gamma, beta, mean, rstd = ctx.saved_tensors
        N, C = x.shape[:2]
        lib = L.lib()
        gy = torch.zeros_like(x) if gy is None else gy.to(x.dtype).contiguous()
        if g_ymean is not None:
            g_ymean = g_ymean.float().contiguous()
        gx = torch.empty_like(x)
        ggamma = torch.empty_like(gamma) if gamma is not None else None
        gbeta = torch.empty_like(beta) if beta is not None else None
        nws = lib.ud_in_act_bwd_workspace_bytes(N, C)
        ws = L.workspace(nws, x.device)
        bwd = lib.ud_in_act_bwd_bf16 if x.dtype == torch.bfloat16 else lib.ud_in_act_bwd
        L.check(bwd(L.ptr(x), L.ptr(gy), L.ptr(gamma), L.ptr(beta), L.ptr(mean), L.ptr(rstd), L.ptr(g_ymean), L.ptr(gx),
                    L.ptr(ggamma), L.ptr(gbeta), L.ptr(ws), ws.numel(), N, C, ctx.hw, ctx.act, L.stream()), "in_act_bwd")
        return gx, ggamma, gbeta, None, None, None


def in_act(x, gamma, beta, act="swish", eps=1e-5, want_mean=False):
    """y = act(instance_norm(x)*gamma+beta); with want_mean also returns y.mean([-2,-1]) [N,C]."""
    y, ymean = _InAct.apply(x, gamma, beta, ACT_CODES[act], eps, want_mean)
    return (y, ymean) if want_mean else y


class _Tanh(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = x.contiguous()
        L.require_cuda_f32(x)
        y = torch.empty_like(x)
        L.check(L.lib().ud_tanh_fwd(L.ptr(x), L.ptr(y), x.numel(), L.stream()), "tanh_fwd")
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, gy):
        (y,) = ctx.saved_tensors
        gy = gy.contiguous()
        gx = torch.empty_like(y)
        L.check(L.lib().ud_tanh_bwd(L.ptr(y), L.ptr(gy), L.ptr(gx), y.numel(), L.stream()), "tanh_bwd")
        return gx


def tanh(x):
    return _Tanh.apply(x)


# ------------------------------------------------------------------------------------------
# a4 / a7: attention() glue
# ------------------------------------------------------------------------------------------
class _BilinearAC(torch.autograd.Function):
    """F.interpolate(mode='bilinear', align_corners=True) (model/unidefense.py:16)."""

    @staticmethod
    def forward(ctx, x, H, W):
        x = x.contiguous()
        L.require_cuda_f32(x)
        h, w = x.shape[-2:]
        planes = x.numel() // (h * w) if h * w else 0
        y = torch.empty(*x.shape[:-2], H, W, device=x.device, dtype=torch.float32)
        L.check(L.lib().ud_bilinear_ac_fwd(L.ptr(x), L.ptr(y), planes, h, w, H, W, L.stream()), "bilinear_fwd")
        ctx.shape = tuple(x.shape)
        return y

    @staticmethod
    def backward(ctx, gy):
        gy = gy.contiguous()
        shape = ctx.shape
        h, w = shape[-2:]
        H, W = gy.shape[-2:]
        gx = torch.empty(shape, device=gy.device, dtype=torch.float32)
        planes = gx.numel() // (h * w) if h * w else 0
        L.check(L.lib().ud_bilinear_ac_bwd(L.ptr(gy), L.ptr(gx), planes, h, w, H, W, L.stream()), "bilinear_bwd")
        return gx, None, None


def bilinear_ac(x, size):
    return _BilinearAC.apply(x, int(size[0]), int(size[1]))


class _AttnPrep(torch.autograd.Function):
    """Error maps (model/unidefense.py:126-134,:148).  Differentiable in x only: the reference passes pred detached
    (dec_out.clone().detach(), :213 / :393 / :586), so no gradient is ever returned for it."""

    @staticmethod
    def forward(ctx, pred, x, h, w, norm_ortho):
        pred = pred.detach().contiguous()
        x = x.detach().contiguous()
        L.require_cuda_f32(pred, x)
        N, C = x.shape[:2]
        sd = torch.empty(N, C, h, w, device=x.device, dtype=torch.float32)
        fd = torch.empty(N, 2 * C, h, w // 2 + 1, device=x.device, dtype=torch.float32)
        L.check(L.lib().ud_attn_prep(L.ptr(pred), L.ptr(x), L.ptr(sd), L.ptr(fd), N, C, pred.shape[-2], pred.shape[-1],
                                     x.shape[-2], x.shape[-1], h, w, norm_ortho, L.stream()), "attn_prep")
        if ctx.needs_input_grad[1]:
            ctx.save_for_backward(pred, x)
        ctx.hw = (h, w)
        ctx.norm_ortho = norm_ortho
        ctx.set_materialize_grads(False)
        return sd, fd

    @staticmethod
    def backward(ctx, g_sd, g_fd):
        if not ctx.needs_input_grad[1] or (g_sd is None and g_fd is None):
            return None, None, None, None, None
        pred, x = ctx.saved_tensors
        N, C = x.shape[:2]
        h, w = ctx.hw
        g_sd = None if g_sd is None else g_sd.contiguous()
        g_fd = None if g_fd is None else g_fd.contiguous()
        g_x = torch.empty_like(x)
        L.check(L.lib().ud_attn_prep_bwd(L.ptr(pred), L.ptr(x), L.ptr(g_sd), L.ptr(g_fd), L.ptr(g_x), N, C,
                                         pred.shape[-2], pred.shape[-1], x.shape[-2], x.shape[-1], h, w, ctx.norm_ortho,
                                         L.stream()), "attn_prep_bwd")
        return None, g_x, None, None, None


def attn_prep(pred, x, size, norm="ortho"):
    """Error maps -> (spat_diff [N,C,h,w], freq_diff [N,2C,h,w/2+1]); differentiable w.r.t. x (pred is data)."""
    return _AttnPrep.apply(pred, x, int(size[0]), int(size[1]), norm_flag(norm))


def _rfft2_raw(x, norm_ortho, adjoint):
    N, C, h, w = x.shape
    xf = torch.empty(N, 2 * C, h, w // 2 + 1, device=x.device, dtype=torch.float32)
    nws = L.lib().ud_rfft2_workspace_bytes(N, C, h, w)          # 0 for the small-plane path (h, w <= 64)
    ws = L.workspace(nws, x.device) if nws else None
    L.check(L.lib().ud_rfft2(L.ptr(x), L.ptr(xf), L.ptr(ws), nws, N, C, h, w, norm_ortho, adjoint, L.stream()), "rfft2_cat")
    return xf


def _irfft2_raw(xf, mask, h, w, norm_ortho, adjoint):
    N, C2 = xf.shape[:2]
    y = torch.empty(N, C2 // 2, h, w, device=xf.device, dtype=torch.float32)
    nws = L.lib().ud_rfft2_workspace_bytes(N, C2 // 2, h, w)
    ws = L.workspace(nws, xf.device) if nws else None
    L.check(L.lib().ud_irfft2(L.ptr(xf), L.ptr(mask), L.ptr(y), L.ptr(ws), nws, N, C2 // 2, h, w, norm_ortho, adjoint,
                              L.stream()), "irfft2_cat")
    return y


class _Rfft2Cat(torch.autograd.Function):
    """cat([re, im], 1) of torch.fft.rfft2 (model/unidefense.py:135-136); backward = fft_r2c_backward."""

    @staticmethod
    def forward(ctx, x, norm_ortho):
        x = x.contiguous()
        L.require_cuda_f32(x)
        ctx.norm_ortho = norm_ortho
        ctx.hw = tuple(x.shape[-2:])
        return _rfft2_raw(x, norm_ortho, 0)

    @staticmethod
    def backward(ctx, g):
        h, w = ctx.hw
        return _irfft2_raw(g.contiguous(), None, h, w, ctx.norm_ortho, 1), None


def rfft2_cat(x, norm="ortho"):
    return _Rfft2Cat.apply(x, norm_flag(norm))


class _Irfft2Cat(torch.autograd.Function):
    """irfft2(complex(*tensor_split(xf, 2, 1)), s=(h, w)) (model/unidefense.py:142-145); backward = fft_c2r_backward."""

    @staticmethod
    def forward(ctx, xf, h, w, norm_ortho):
        xf = xf.contiguous()
        L.require_cuda_f32(xf)
        if xf.shape[-2] != h or xf.shape[-1] != w // 2 + 1 or xf.shape[1] % 2:
            raise ValueError(f"irfft2_cat: spectrum {tuple(xf.shape)} does not match s=({h},{w})")
        ctx.norm_ortho = norm_ortho
        return _irfft2_raw(xf, None, h, w, norm_ortho, 0)

    @staticmethod
    def backward(ctx, gy):
        return _rfft2_raw(gy.contiguous(), ctx.norm_ortho, 1), None, None, None


def irfft2_cat(xf, size, norm="ortho"):
    return _Irfft2Cat.apply(xf, int(size[0]), int(size[1]), norm_flag(norm))


def spectral_mask_filter(x, mask, norm="ortho"):
    """y = irfft2(mask * rfft2(x)) for any plane size (no grad): the composite of BASELINE.json's frequency-branch
    microbench (configs[4]: batched FFT2 + mask + IFFT2).  x [N,C,H,W]; mask [N,H,W/2+1] is shared by the channels of a
    sample, as the dynamic filter's mask is (model/unidefense.py:140-145).  Two generic transforms (csrc/ud_fft2d.cu);
    the mask multiply rides on the inverse transform's load."""
    x = x.detach().contiguous()
    mask = mask.detach().contiguous()
    L.require_cuda_f32(x, mask)
    N, C, H, W = x.shape
    if tuple(mask.shape) != (N, H, W // 2 + 1):
        raise ValueError(f"spectral_mask_filter: mask {tuple(mask.shape)} does not match [N,H,W/2+1] of {tuple(x.shape)}")
    nf = norm_flag(norm)
    return _irfft2_raw(_rfft2_raw(x, nf, 0), mask, H, W, nf, 0)


class _AttnFuse(torch.autograd.Function):
    """out = (1-s)*smask*emb + s*ff + res, s = sigmoid(fuse_coef) (model/unidefense.py:153-155).
    res=None means the residual is emb itself (dropout inactive)."""

    @staticmethod
    def forward(ctx, emb, smask, ff, res, fuse_coef):
        emb, smask, ff = emb.contiguous(), smask.contiguous(), ff.contiguous()
        res = None if res is None else res.contiguous()
        coef = fuse_coef.reshape(1).contiguous()
        L.require_cuda_f32(emb, smask, ff, res, coef)
        N, C = emb.shape[:2]
        HW = emb.shape[2] * emb.shape[3]
        out = torch.empty_like(emb)
        L.check(L.lib().ud_attn_fuse_fwd(L.ptr(emb), L.ptr(smask), L.ptr(ff), L.ptr(res), L.ptr(coef), L.ptr(out),
                                         N, C, HW, L.stream()), "attn_fuse_fwd")
        ctx.save_for_backward(emb, smask, ff, coef)
        ctx.res_is_emb = res is None
        ctx.coef_shape = fuse_coef.shape
        return out

    @staticmethod
    def backward(ctx, g):
        emb, smask, ff, coef = ctx.saved_tensors
        g = g.contiguous()
        N, C = emb.shape[:2]
        HW = emb.shape[2] * emb.shape[3]
        lib = L.lib()
        g_emb, g_ff = torch.empty_like(emb), torch.empty_like(ff)
        g_smask = torch.empty_like(smask)
        g_coef = torch.empty(1, device=emb.device, dtype=torch.float32)
        ws = L.workspace(lib.ud_attn_fuse_bwd_workspace_bytes(N, HW), emb.device)
        L.check(lib.ud_attn_fuse_bwd(L.ptr(emb), L.ptr(smask), L.ptr(ff), L.ptr(g), L.ptr(coef), L.ptr(g_emb),
                                     L.ptr(g_ff), L.ptr(g_smask), L.ptr(g_coef), L.ptr(ws), ws.numel(), N, C, HW,
                                     int(ctx.res_is_emb), L.stream()), "attn_fuse_bwd")
        return g_emb, g_smask, g_ff, (None if ctx.res_is_emb else g), g_coef.reshape(ctx.coef_shape)


def attn_fuse(emb, smask, ff, res, fuse_coef):
    return _AttnFuse.apply(emb, smask, ff, res, fuse_coef)


# ------------------------------------------------------------------------------------------
# a5 / a6: dynamic filters -- everything after layer1's conv
# ------------------------------------------------------------------------------------------
def bn_local_stats(proj):
    """-> (mean [C], m2 [C]) of proj [N,C,h,w] over (N,h,w); m2 = sum (x-mean)^2."""
    N, C = proj.shape[:2]
    HW = proj.shape[2] * proj.shape[3]
    mean = torch.empty(C, device=proj.device, dtype=torch.float32)
    m2 = torch.empty(C, device=proj.device, dtype=torch.float32)
    L.check(L.lib().ud_bn_stats(L.ptr(proj), L.ptr(mean), L.ptr(m2), N, C, HW, L.stream()), "bn_stats")
    return mean, m2


def proj_precision():
    """Arithmetic of the tcgen05 projections: plain TF32 when torch would let cuDNN use TF32 for convolutions
    (torch's default), otherwise 3xTF32 (hi/lo operand split, fp32-grade accuracy)."""
    return "tf32" if torch.backends.cudnn.allow_tf32 else "3xtf32"


def proj_supported(x, conv):
    """Shapes the tcgen05 implicit GEMM takes (include/unidefense_b200.h: ud_proj_fwd); anything else stays on
    the library convolution."""
    k = conv.kernel_size
    return (x.is_cuda and x.dim() == 4 and conv.bias is None and conv.groups == 1 and k[0] == k[1] and k[0] in (1, 3)
            and tuple(conv.stride) == (1, 1) and tuple(conv.dilation) == (1, 1)
            and tuple(conv.padding) == (k[0] // 2, k[0] // 2) and conv.padding_mode == "zeros"
            and conv.in_channels % 4 == 0 and conv.in_channels >= 32 and x.shape[-1] <= 128)


class _ProjConv(torch.autograd.Function):
    """Bias-free 1x1 / 3x3 (pad 1) convolution = FrequencyDynamicFilter.layer1[0] / SpatialDynamicFilter.layer1[0]
    (model/modules.py:82-85, :111-114) on tcgen05, returning the BatchNorm batch statistics of its output
    (mean [Cout], m2 [Cout]) from the GEMM epilogue.  Backward: the library's convolution_backward."""

    @staticmethod
    def forward(ctx, x, weight, precision, want_stats):
        if not weight.is_cuda or weight.dtype != torch.float32:
            raise RuntimeError("proj_conv: weight must be a CUDA fp32 tensor (no CPU fallback)")
        if x.dtype != torch.float32 or not x.is_cuda:
            raise RuntimeError("proj_conv: x must be a CUDA fp32 tensor (no CPU fallback)")
        N, Cin, H, W = x.shape
        Cout, _, k, _ = weight.shape
        lib = L.lib()
        dev = x.device
        split = precision == "3xtf32"
        if precision not in ("tf32", "3xtf32"):
            raise ValueError(f"proj_conv: precision {precision!r} (tf32 | 3xtf32)")
        nhwc = x.is_contiguous(memory_format=torch.channels_last) and not x.is_contiguous()
        if nhwc and not split:
            x_hi, x_lo = x, None                       # already [N,H,W,C] in memory
        else:
            xc = x.contiguous()
            x_hi = torch.empty(N, H, W, Cin, device=dev, dtype=torch.float32)
            x_lo = torch.empty_like(x_hi) if split else None
            L.check(lib.ud_proj_prep_x(L.ptr(xc), L.ptr(x_hi), L.ptr(x_lo), N, Cin, H * W, L.stream()), "proj_prep_x")
        w_cl = k > 1 and weight.is_contiguous(memory_format=torch.channels_last)
        wc = weight if w_cl else weight.contiguous()
        if not split and (k == 1 or w_cl):
            w_hi, w_lo = wc, None                      # [Cout, Cin] / channels_last [Cout, ky, kx, Cin]: already K-major
        elif w_cl:                                     # split a K-major weight: taps = 1 re-layout is the identity
            w_hi = torch.empty(Cout, k * k, Cin, device=dev, dtype=torch.float32)
            w_lo = torch.empty_like(w_hi)
            L.check(lib.ud_proj_prep_w(L.ptr(wc), L.ptr(w_hi), L.ptr(w_lo), Cout, k * k * Cin, 1, L.stream()), "proj_prep_w")
        else:
            w_hi = torch.empty(Cout, k * k, Cin, device=dev, dtype=torch.float32)
            w_lo = torch.empty_like(w_hi) if split else None
            L.check(lib.ud_proj_prep_w(L.ptr(wc), L.ptr(w_hi), L.ptr(w_lo), Cout, Cin, k * k, L.stream()), "proj_prep_w")
        y = torch.empty(N, Cout, H, W, device=dev, dtype=torch.float32)
        tiles = lib.ud_proj_m_tiles(N, H, W, k)
        if tiles < 0:
            raise RuntimeError("proj_conv: " + lib.ud_last_error().decode(errors="replace"))
        pm = p2 = pc = mean = m2 = None
        if want_stats:
            pm = torch.empty(tiles, Cout, device=dev, dtype=torch.float32)
            p2 = torch.empty_like(pm)
            pc = torch.empty(tiles, device=dev, dtype=torch.float32)
        L.check(lib.ud_proj_fwd(L.ptr(x_hi), L.ptr(x_lo), L.ptr(w_hi), L.ptr(w_lo), L.ptr(y), L.ptr(pm), L.ptr(p2),
                                L.ptr(pc), N, H, W, Cin, Cout, k, L.stream()), "proj_fwd")
        if want_stats:
            mean = torch.empty(Cout, device=dev, dtype=torch.float32)
            m2 = torch.empty_like(mean)
            L.check(lib.ud_bn_merge_partials(L.ptr(pm), L.ptr(p2), L.ptr(pc), L.ptr(mean), L.ptr(m2), tiles, Cout,
                                             L.stream()), "bn_merge_partials")
            ctx.mark_non_differentiable(mean, m2)
        ctx.save_for_backward(x, weight)
        ctx.k = k
        ctx.split = split
        return y, mean, m2

    @staticmethod
    def backward(ctx, gy, _gm, _g2):
        """Data gradient (1x1 and 3x3) and the 1x1 weight gradient on the same tcgen05 kernel; the 3x3 weight gradient
        (and shapes outside the kernel's limits) through the library's convolution_backward."""
        x, weight = ctx.saved_tensors
        k, split = ctx.k, ctx.split
        N, Cin, H, W = x.shape
        Cout = weight.shape[0]
        lib = L.lib()
        dev = x.device
        gy = gy.contiguous()
        need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gx = gw = None
        if need_x and Cout % 4 == 0 and Cout >= 32:
            g_hi = torch.empty(N, H, W, Cout, device=dev, dtype=torch.float32)
            g_lo = torch.empty_like(g_hi) if split else None
            L.check(lib.ud_proj_prep_x(L.ptr(gy), L.ptr(g_hi), L.ptr(g_lo), N, Cout, H * W, L.stream()), "proj_prep_x")
            wc = weight.contiguous()
            wt_hi = torch.empty(Cin, k * k, Cout, device=dev, dtype=torch.float32)
            wt_lo = torch.empty_like(wt_hi) if split else None
            L.check(lib.ud_proj_prep_wt(L.ptr(wc), L.ptr(wt_hi), L.ptr(wt_lo), Cout, Cin, k * k, L.stream()), "proj_prep_w")
            gx = torch.empty(N, Cin, H, W, device=dev, dtype=torch.float32)
            L.check(lib.ud_proj_fwd(L.ptr(g_hi), L.ptr(g_lo), L.ptr(wt_hi), L.ptr(wt_lo), L.ptr(gx), None, None, None,
                                    N, H, W, Cout, Cin, k, L.stream()), "proj_dgrad")
            need_x = False
        if need_w and k == 1 and (H * W) % 4 == 0 and H * W >= 32:
            xc = x.contiguous()
            if split:
                x_hi, x_lo, d_hi, d_lo = (torch.empty_like(xc), torch.empty_like(xc), torch.empty_like(gy), torch.empty_like(gy))
                L.check(lib.ud_proj_split(L.ptr(xc), L.ptr(x_hi), L.ptr(x_lo), xc.numel(), L.stream()), "proj_prep_x")
                L.check(lib.ud_proj_split(L.ptr(gy), L.ptr(d_hi), L.ptr(d_lo), gy.numel(), L.stream()), "proj_prep_x")
            else:
                x_hi, x_lo, d_hi, d_lo = xc, None, gy, None
            gw = torch.empty(Cout, Cin, 1, 1, device=dev, dtype=torch.float32)
            L.check(lib.ud_proj_wgrad_1x1(L.ptr(x_hi), L.ptr(x_lo), L.ptr(d_hi), L.ptr(d_lo), L.ptr(gw), N, H * W, Cin, Cout,
                                          L.stream()), "proj_wgrad")
            need_w = False
        if need_x or need_w:
            ax, aw, _ = torch.ops.aten.convolution_backward(gy, x, weight, None, [1, 1], [k // 2, k // 2], [1, 1], False,
                                                            [0, 0], 1, [need_x, need_w, False])
            gx = ax if need_x else gx
            gw = aw if need_w else gw
        return gx, gw, None, None


def proj_conv(x, weight, precision=None, want_stats=True):
    """-> (y [N,Cout,H,W] NCHW fp32, mean [Cout] | None, m2 [Cout] | None)."""
    return _ProjConv.apply(x, weight, precision or proj_precision(), bool(want_stats))


class _DyfiMask(torch.autograd.Function):
    """BN-apply + act + channel mean/max + cat(diff) + conv1x1 + sigmoid (+ mask*x)
    (model/modules.py:94-104, :123-133).  mean/rstd are the (possibly cross-rank) BN statistics;
    `count` = global N*h*w in training (batch statistics take part in the backward), 0 in eval.
    `stat_reduce` (optional callable) sums a [2, C] tensor over ranks (SyncBatchNorm backward)."""

    @staticmethod
    def forward(ctx, proj, mean, rstd, gamma, beta, diff, w2, x, act, count, want_out, stat_reduce):
        proj, diff = proj.contiguous(), diff.contiguous()
        x = x.contiguous()
        w2f = w2.reshape(-1).contiguous()
        L.require_cuda_f32(proj, mean, rstd, gamma, beta, diff, w2f, x)
        N, Cp, h, w = proj.shape
        HW, D, Cx = h * w, diff.shape[1], x.shape[1]
        if w2f.numel() != 2 + D:
            raise ValueError(f"dyfi_mask: layer2 weight has {w2f.numel()} inputs, expected {2 + D}")
        dev = proj.device
        mask = torch.empty(N, 1, h, w, device=dev, dtype=torch.float32)
        out = torch.empty_like(x) if want_out else None
        pmean = torch.empty(N, HW, device=dev, dtype=torch.float32)
        pmax = torch.empty(N, HW, device=dev, dtype=torch.float32)
        argmax = torch.empty(N, HW, device=dev, dtype=torch.int32)
        L.check(L.lib().ud_dyfi_mask_fwd(L.ptr(proj), L.ptr(mean), L.ptr(rstd), L.ptr(gamma), L.ptr(beta), L.ptr(diff),
                                         L.ptr(w2f), L.ptr(x), L.ptr(mask), L.ptr(out), L.ptr(pmean), L.ptr(pmax),
                                         L.ptr(argmax), N, Cp, D, Cx, HW, act, L.stream()), "dyfi_mask_fwd")
        ctx.save_for_backward(proj, mean, rstd, gamma, beta, diff, w2f, x, mask, pmean, pmax, argmax)
        ctx.act, ctx.count, ctx.want_out, ctx.stat_reduce = act, count, want_out, stat_reduce
        ctx.w2_shape = w2.shape
        if want_out:
            return mask, out
        return mask, None

    @staticmethod
    def backward(ctx, g_mask, g_out):
        proj, mean, rstd, gamma, beta, diff, w2f, x, mask, pmean, pmax, argmax = ctx.saved_tensors
        N, Cp, h, w = proj.shape
        HW, D, Cx = h * w, diff.shape[1], x.shape[1]
        lib = L.lib()
        dev = proj.device
        g_mask = None if g_mask is None else g_mask.contiguous()
        g_out = None if (g_out is None or not ctx.want_out) else g_out.contiguous()
        g_x = torch.empty_like(x) if g_out is not None else None
        dz = torch.empty_like(proj)
        g_w2 = torch.empty(2 + D, device=dev, dtype=torch.float32)
        ws = L.workspace(lib.ud_dyfi_mask_bwd_workspace_bytes(N, HW), dev)
        # the error maps carry x's gradient (model/modules.py:101-103, :130-132)
        g_diff = torch.empty_like(diff) if ctx.needs_input_grad[5] else None
        L.check(lib.ud_dyfi_mask_bwd(L.ptr(proj), L.ptr(mean), L.ptr(rstd), L.ptr(gamma), L.ptr(beta), L.ptr(diff),
                                     L.ptr(w2f), L.ptr(x), L.ptr(mask), L.ptr(pmean), L.ptr(pmax), L.ptr(argmax),
                                     L.ptr(g_mask), L.ptr(g_out), L.ptr(g_x), L.ptr(dz), L.ptr(g_w2), L.ptr(g_diff),
                                     L.ptr(ws), ws.numel(), N, Cp, D, Cx, HW, ctx.act, L.stream()), "dyfi_mask_bwd")
        sums = torch.empty(2, Cp, device=dev, dtype=torch.float32)
        L.check(lib.ud_bn_bwd_reduce(L.ptr(dz), L.ptr(proj), L.ptr(mean), L.ptr(rstd), L.ptr(sums[0]), L.ptr(sums[1]),
                                     N, Cp, HW, L.stream()), "bn_bwd_reduce")
        g_beta, g_gamma = sums[0].clone(), sums[1].clone()      # local sums: DDP averages parameter grads
        count = ctx.count
        training = torch.is_tensor(count) or bool(count)
        if ctx.stat_reduce is not None and training:
            sums = ctx.stat_reduce(sums)
        g_proj = torch.empty_like(proj)
        if torch.is_tensor(count):           # cross-rank count lives on the device: fold 1/count into the sums
            sums = sums / count
            inv_count = 1.0
        else:
            inv_count = 1.0 / count if count else 0.0
        L.check(lib.ud_bn_bwd_apply(L.ptr(dz), L.ptr(proj), L.ptr(mean), L.ptr(rstd), L.ptr(gamma), L.ptr(sums[0]),
                                    L.ptr(sums[1]), inv_count, L.ptr(g_proj), N, Cp, HW, L.stream()), "bn_bwd_apply")
        return (g_proj, None, None, g_gamma if gamma is not None else None, g_beta if beta is not None else None,
                g_diff, g_w2.reshape(ctx.w2_shape), g_x, None, None, None, None)


def dyfi_mask(proj, mean, rstd, gamma, beta, diff, w2, x, act="swish", count=0, want_out=True, stat_reduce=None):
    """-> (mask [N,1,h,w], out = mask*x or None)."""
    return _DyfiMask.apply(proj, mean, rstd, gamma, beta, diff, w2, x, ACT_CODES[act],
                           count if torch.is_tensor(count) else int(count), bool(want_out), stat_reduce)


# ------------------------------------------------------------------------------------------
# a9-a11: losses (forward also produces the gradient; backward is a scalar multiply)
# ------------------------------------------------------------------------------------------
class _Triplet(torch.autograd.Function):
    """AsymmetricalWeightedTripletLoss.forward (loss/triplet_loss.py:75-82)."""

    @staticmethod
    def forward(ctx, feat, labels):
        feat = feat.contiguous()
        L.require_cuda_f32(feat)
        if labels.dtype != torch.int64 or not labels.is_cuda:
            raise RuntimeError("triplet: labels must be a CUDA int64 tensor")
        labels = labels.contiguous()
        N, c = feat.shape
        if labels.numel() != N:
            raise ValueError("triplet: labels/feat batch mismatch")
        loss = torch.empty((), device=feat.device, dtype=torch.float32)
        g = torch.empty_like(feat) if ctx.needs_input_grad[0] else None
        L.check(L.lib().ud_triplet_fwd(L.ptr(feat), L.ptr(labels), L.ptr(loss), L.ptr(g), N, c, L.stream()), "triplet")
        ctx.save_for_backward(g)
        return loss

    @staticmethod
    def backward(ctx, gl):
        (g,) = ctx.saved_tensors
        return g * gl, None


def triplet_loss(feat, labels):
    return _Triplet.apply(feat, labels)


class _Factorization(torch.autograd.Function):
    """FactorizationLoss.forward (loss/calib_loss.py:17-28)."""

    @staticmethod
    def forward(ctx, a, b, off_w, eps):
        if ctx.needs_input_grad[1]:
            raise RuntimeError("factorization_loss: only emb_a is differentiated (the engine passes emb_b detached, "
                               "engine/abstract_engine.py:230); detach emb_b or swap the arguments")
        a, b = a.contiguous(), b.detach().contiguous()
        L.require_cuda_f32(a, b)
        N, F_ = a.shape
        if tuple(b.shape) != (N, F_):
            raise ValueError("factorization: emb_a / emb_b shapes differ")
        lib = L.lib()
        loss = torch.empty((), device=a.device, dtype=torch.float32)
        g = torch.empty_like(a) if ctx.needs_input_grad[0] else None
        ws = L.workspace(lib.ud_factorization_workspace_bytes(N, F_), a.device)
        L.check(lib.ud_factorization_fwd(L.ptr(a), L.ptr(b), L.ptr(loss), L.ptr(g), L.ptr(ws), ws.numel(), N, F_,
                                         float(off_w), float(eps), L.stream()), "factorization")
        ctx.save_for_backward(g)
        return loss

    @staticmethod
    def backward(ctx, gl):
        (g,) = ctx.saved_tensors
        return g * gl, None, None, None


def factorization_loss(emb_a, emb_b, off_diag_weight=0.005, eps=1e-6):
    return _Factorization.apply(emb_a, emb_b, off_diag_weight, eps)


class _MaskKL(torch.autograd.Function):
    """fused=True: KLDivLoss(batchmean, log_target)(log_softmax(pred.flat), log_softmax(gt.flat))
    (engine/abstract_engine.py:333-346).  fused=False: the bare KLDivLoss on log-probabilities."""

    @staticmethod
    def forward(ctx, pred, gt, fused=True):
        if ctx.needs_input_grad[1]:
            raise RuntimeError("mask KL: the target is not differentiated (the engine detaches it, "
                               "engine/abstract_engine.py:215-228); detach it")
        shape = pred.shape
        N = shape[0]
        p = pred.reshape(N, -1).contiguous()
        q = gt.detach().reshape(N, -1).contiguous()
        L.require_cuda_f32(p, q)
        lib = L.lib()
        loss = torch.empty((), device=p.device, dtype=torch.float32)
        g = torch.empty_like(p) if ctx.needs_input_grad[0] else None
        ws = L.workspace(lib.ud_mask_kl_workspace_bytes(N), p.device)
        fn = lib.ud_mask_kl_fwd if fused else lib.ud_kl_div_log_target_fwd
        L.check(fn(L.ptr(p), L.ptr(q), L.ptr(loss), L.ptr(g), L.ptr(ws), ws.numel(), N, p.shape[1], L.stream()),
                "mask_kl" if fused else "kl_div")
        ctx.save_for_backward(g)
        ctx.shape = shape
        return loss

    @staticmethod
    def backward(ctx, gl):
        (g,) = ctx.saved_tensors
        return (g * gl).reshape(ctx.shape), None, None


def mask_kl_loss(mask_pred, mask_gt):
    return _MaskKL.apply(mask_pred, mask_gt, True)


def kl_div_log_target(log_pred, log_target):
    """nn.KLDivLoss(reduction='batchmean', log_target=True)(log_pred, log_target) for [N, M] inputs."""
    return _MaskKL.apply(log_pred, log_target, False)


class _CrossEntropy(torch.autograd.Function):
    """nn.CrossEntropyLoss() / nn.BCEWithLogitsLoss() as the engine calls them (engine/abstract_engine.py:256-259)."""

    @staticmethod
    def forward(ctx, logits, target, binary):
        logits = logits.contiguous()
        L.require_cuda_f32(logits)
        loss = torch.empty((), device=logits.device, dtype=torch.float32)
        g = torch.empty_like(logits) if ctx.needs_input_grad[0] else None
        lib = L.lib()
        if binary:
            t = target.detach().to(torch.float32).contiguous()
            if t.shape != logits.shape:
                raise ValueError(f"bce_with_logits: logits {tuple(logits.shape)} vs target {tuple(t.shape)}")
            L.check(lib.ud_bce_with_logits_fwd(L.ptr(logits), L.ptr(t), L.ptr(loss), L.ptr(g), logits.numel(), L.stream()),
                    "bce_with_logits")
        else:
            if target.dtype != torch.int64 or not target.is_cuda or logits.dim() != 2 or target.numel() != logits.shape[0]:
                raise RuntimeError("cross_entropy: logits [N,K] fp32 and CUDA int64 class targets [N] expected")
            L.check(lib.ud_cross_entropy_fwd(L.ptr(logits), L.ptr(target.contiguous()), L.ptr(loss), L.ptr(g),
                                             logits.shape[0], logits.shape[1], L.stream()), "cross_entropy")
        ctx.save_for_backward(g)
        return loss

    @staticmethod
    def backward(ctx, gl):
        (g,) = ctx.saved_tensors
        return g * gl, None, None


def cross_entropy(logits, target):
    return _CrossEntropy.apply(logits.float(), target, False)


def bce_with_logits(logits, target):
    return _CrossEntropy.apply(logits.float(), target, True)


# ------------------------------------------------------------------------------------------
# a13-a16: perturbations (blur and downscale are differentiable, as in the reference; the style transfers and coral
# run under no_grad there, model/unidefense.py:181-193, and here)
# ------------------------------------------------------------------------------------------
class _Blur5(torch.autograd.Function):
    """random_blur (model/modules.py:15-16); backward = the adjoint 5x5 stencil with the reflected taps folded back."""

    @staticmethod
    def forward(ctx, x):
        x = x.detach().contiguous()
        L.require_cuda_f32(x)
        H, W = x.shape[-2:]
        y = torch.empty_like(x)
        L.check(L.lib().ud_gaussian_blur5(L.ptr(x), L.ptr(y), x.numel() // (H * W), H, W, L.stream()), "gaussian_blur5")
        return y

    @staticmethod
    def backward(ctx, gy):
        gy = gy.contiguous()
        H, W = gy.shape[-2:]
        gx = torch.empty_like(gy)
        L.check(L.lib().ud_gaussian_blur5_bwd(L.ptr(gy), L.ptr(gx), gy.numel() // (H * W), H, W, L.stream()),
                "gaussian_blur5_bwd")
        return gx


def gaussian_blur5(x):
    """random_blur (model/modules.py:15-16)."""
    return _Blur5.apply(x)


class _Downscale(torch.autograd.Function):
    """downscale (model/modules.py:19-21); backward = sum over each input pixel's nearest-index preimage."""

    @staticmethod
    def forward(ctx, x, bottleneck_scale):
        x = x.detach().contiguous()
        L.require_cuda_f32(x)
        H, W = x.shape[-2:]
        y = torch.empty_like(x)
        L.check(L.lib().ud_downscale_nearest(L.ptr(x), L.ptr(y), x.numel() // (H * W), H, W, bottleneck_scale,
                                             L.stream()), "downscale")
        ctx.scale = bottleneck_scale
        return y

    @staticmethod
    def backward(ctx, gy):
        gy = gy.contiguous()
        H, W = gy.shape[-2:]
        gx = torch.empty_like(gy)
        L.check(L.lib().ud_downscale_nearest_bwd(L.ptr(gy), L.ptr(gx), gy.numel() // (H * W), H, W, ctx.scale,
                                                 L.stream()), "downscale_bwd")
        return gx, None


def downscale_nearest(x, bottleneck_scale=0.75):
    """downscale (model/modules.py:19-21)."""
    return _Downscale.apply(x, float(bottleneck_scale))


def freq_style_transfer(content, style, lmda):
    """FrequencyStyleTransfer (model/modules.py:43-54); lmda [B] in [0.5, 1).  Fused rows / cols+mix / rows^-1
    kernels, spectra stay in an L2-resident workspace."""
    content, style = content.detach().contiguous(), style.detach().contiguous()
    lm = lmda.detach().reshape(-1).to(device=content.device, dtype=torch.float32).contiguous()
    L.require_cuda_f32(content, style, lm)
    if content.shape != style.shape or lm.numel() != content.shape[0]:
        raise ValueError("freq_style_transfer: content/style/lmda shapes disagree")
    N, C, H, W = content.shape
    lib = L.lib()
    out = torch.empty_like(content)
    ws = L.workspace(lib.ud_freq_style_workspace_bytes(N, C, H, W), content.device)
    L.check(lib.ud_freq_style_transfer(L.ptr(content), L.ptr(style), L.ptr(lm), L.ptr(out), L.ptr(ws), ws.numel(), N, C,
                                       H, W, L.stream()), "freq_style_transfer")
    return out


def spatial_style_transfer(content, style, lmda):
    """SpatialStyleTransfer (model/modules.py:59-76): exact histogram (rank) matching per (n, c) plane; lmda [B].
    One stable radix sort per plane with the blend fused into the last pass (csrc/ud_style_sort.cu) instead of the
    reference's two torch.sort + argsort + gather."""
    content, style = content.detach().contiguous(), style.detach().contiguous()
    L.require_cuda_f32(content, style)
    if content.shape != style.shape or content.dim() != 4:
        raise AssertionError(f"spatial_style_transfer: content {tuple(content.shape)} and style {tuple(style.shape)} "
                             "must share one [B,C,H,W] shape")          # the reference asserts (modules.py:61)
    B, C, H, W = content.shape
    lm = lmda.detach().reshape(-1).to(device=content.device, dtype=torch.float32).contiguous()
    if lm.numel() != B:
        raise ValueError(f"spatial_style_transfer: lmda has {lm.numel()} entries for a batch of {B}")
    out = torch.empty_like(content)
    lib = L.lib()
    nws = lib.ud_spatial_style_workspace_bytes(B, C, H * W)
    ws = L.workspace(nws, content.device)
    L.check(lib.ud_spatial_style_transfer(L.ptr(content), L.ptr(style), L.ptr(lm), L.ptr(out), L.ptr(ws), nws, B, C, H * W,
                                          L.stream()), "spatial_style")
    return out


def coral_batch(source, target):
    """coral (utils/operation.py:20-45) for every (source[n], target[n]) pair in three launches (csrc/ud_coral.cu): the
    per-sample Python loop of model/unidefense.py:189-191 and its 2N host-synchronising 3x3 SVDs are gone.  The
    reference's 'square root' U*sqrt(D)*Vh^T (Appendix D) depends on the sign convention of the SVD library; the
    kernel fixes the gauge (largest component of each eigenvector positive) and parity is asserted modulo it."""
    source, target = source.detach().contiguous(), target.detach().contiguous()
    L.require_cuda_f32(source, target)
    if source.shape != target.shape or source.dim() != 4 or source.shape[1] != 3:
        raise ValueError(f"coral_batch: expected two [N,3,H,W] tensors, got {tuple(source.shape)} / {tuple(target.shape)}")
    N, _, H, W = source.shape
    lib = L.lib()
    out = torch.empty_like(source)
    ws = L.workspace(lib.ud_coral_workspace_bytes(N, H * W), source.device)
    L.check(lib.ud_coral(L.ptr(source), L.ptr(target), L.ptr(out), L.ptr(ws), ws.numel(), N, H * W, L.stream()), "coral")
    return out


# ------------------------------------------------------------------------------------------
# a17 (next row, first step): glue kernels of the SFConv frequency branch
# ------------------------------------------------------------------------------------------
def _fmt(t):
    """-> (nhwc, bf16) of a 4-D activation; anything else is made NCHW-contiguous fp32 by the caller."""
    nhwc = t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous()
    return int(nhwc), int(t.dtype == torch.bfloat16)


class _SfPack(torch.autograd.Function):
    """complex64 spectrum [N,C,h,wh] -> planar cat([re, im], 1) [N,2C,h,wh] in `dtype` / `channels_last`."""

    @staticmethod
    def forward(ctx, spec, dtype, channels_last):
        spec = spec.contiguous()
        if not spec.is_cuda or spec.dtype != torch.complex64:
            raise RuntimeError("sf_pack needs a CUDA complex64 spectrum (no CPU fallback)")
        N, C, h, wh = spec.shape
        nhwc = int(bool(channels_last) and C % 2 == 0)
        planar = torch.empty(N, 2 * C, h, wh, device=spec.device, dtype=dtype,
                             memory_format=torch.channels_last if nhwc else torch.contiguous_format)
        L.check(L.lib().ud_sf_pack(L.ptr(spec), L.ptr(planar), N, C, h * wh, nhwc, int(dtype == torch.bfloat16),
                                   L.stream()), "sf_pack")
        return planar

    @staticmethod
    def backward(ctx, g):
        return _sf_unpack_raw(g), None, None


def _sf_unpack_raw(planar):
    N, C2, h, wh = planar.shape
    C = C2 // 2
    if planar.dtype not in (torch.float32, torch.bfloat16):
        planar = planar.float()
    nhwc, bf16 = _fmt(planar)
    if not nhwc:
        planar = planar.contiguous()
    elif C % 2:
        planar, nhwc = planar.contiguous(), 0
    spec = torch.empty(N, C, h, wh, device=planar.device, dtype=torch.complex64)
    L.check(L.lib().ud_sf_unpack(L.ptr(planar), L.ptr(spec), N, C, h * wh, nhwc, bf16, L.stream()), "sf_unpack")
    return spec


class _SfUnpack(torch.autograd.Function):
    """planar [N,2C,h,wh] (fp32|bf16, NCHW|channels-last) -> complex64 [N,C,h,wh]."""

    @staticmethod
    def forward(ctx, planar):
        if not planar.is_cuda:
            raise RuntimeError("sf_unpack needs CUDA tensors (no CPU fallback)")
        ctx.dtype = planar.dtype
        ctx.cl = bool(_fmt(planar)[0])
        return _sf_unpack_raw(planar)

    @staticmethod
    def backward(ctx, g):
        return _SfPack.apply(g, ctx.dtype, ctx.cl)


def sf_pack(spec, dtype=torch.float32, channels_last=False):
    return _SfPack.apply(spec, dtype, channels_last)


def sf_unpack(planar):
    return _SfUnpack.apply(planar)


class _SfMix(torch.autograd.Function):
    """(1 - sigmoid(coef)) * spat + sigmoid(coef) * freq; spat in the convolution's dtype/layout, freq fp32 NCHW."""

    @staticmethod
    def forward(ctx, spat, freq, coef):
        if not spat.is_cuda:
            raise RuntimeError("sf_mix needs CUDA tensors (no CPU fallback)")
        if spat.dtype not in (torch.float32, torch.bfloat16):
            spat = spat.float()
        nhwc, bf16 = _fmt(spat)
        N, C = spat.shape[:2]
        if nhwc and C % 2:
            nhwc = 0
        if not nhwc:
            spat = spat.contiguous()
        freq = freq.contiguous()
        c = coef.reshape(1).contiguous()
        L.require_cuda_f32(freq, c)
        P = spat.shape[2] * spat.shape[3]
        out = torch.empty_like(spat)
        L.check(L.lib().ud_sf_mix_fwd(L.ptr(spat), L.ptr(freq), L.ptr(c), L.ptr(out), N, C, P, nhwc, bf16, L.stream()),
                "sf_mix_fwd")
        ctx.save_for_backward(spat, freq, c)
        ctx.fmt = (nhwc, bf16)
        ctx.coef_shape = coef.shape
        return out

    @staticmethod
    def backward(ctx, g):
        spat, freq, c = ctx.saved_tensors
        nhwc, bf16 = ctx.fmt
        N, C = spat.shape[:2]
        P = spat.shape[2] * spat.shape[3]
        g = g.to(spat.dtype)
        g = g.contiguous(memory_format=torch.channels_last) if nhwc else g.contiguous()
        lib = L.lib()
        g_spat = torch.empty_like(spat)
        g_freq = torch.empty_like(freq)
        g_coef = torch.empty(1, device=spat.device, dtype=torch.float32)
        ws = L.workspace(lib.ud_sf_mix_bwd_workspace_bytes(N, C, P), spat.device)
        L.check(lib.ud_sf_mix_bwd(L.ptr(g), L.ptr(spat), L.ptr(freq), L.ptr(c), L.ptr(g_spat), L.ptr(g_freq), L.ptr(g_coef),
                                  L.ptr(ws), ws.numel(), N, C, P, nhwc, bf16, L.stream()), "sf_mix_bwd")
        return g_spat, g_freq, g_coef.reshape(ctx.coef_shape)


def sf_mix(spat, freq, coef):
    return _SfMix.apply(spat, freq, coef)


# ------------------------------------------------------------------------------------------
# a19: projected-gradient attack step (unidefense_b200/attack.py)
# ------------------------------------------------------------------------------------------
ATTACK_NORMS = {"linf": 0, "l2": 2}


def attack_step(x0, x_adv, g, loss, best_loss, x_best, eps, alpha, lo, hi, norm="linf"):
    """One PGD iteration in place (csrc/ud_attack.cu): best-iterate select of x_adv by `loss`, then (unless g is None)
    the step under `norm` ('linf' | 'l2'), the projection onto the eps-ball around x0 and the clamp to [lo, hi].
    x0, x_adv, g, x_best: fp32 [N, ...] of one shape; loss, best_loss, eps, alpha: fp32 [N] (eps / alpha may be None
    for a select-only call).  Updates x_adv, best_loss and x_best; the attack state is not differentiated."""
    if norm not in ATTACK_NORMS:
        raise ValueError(f"attack_step: norm must be one of {sorted(ATTACK_NORMS)}, got {norm!r}")
    L.require_cuda_f32(x0, x_adv, g, loss, best_loss, x_best, eps, alpha)
    N = x0.shape[0]
    if x_adv.shape != x0.shape or x_best.shape != x0.shape or (g is not None and g.shape != x0.shape):
        raise ValueError("attack_step: x0, x_adv, g and x_best must share one shape")
    for name, t in (("loss", loss), ("best_loss", best_loss), ("eps", eps), ("alpha", alpha)):
        if t is not None and t.numel() != N:
            raise ValueError(f"attack_step: {name} has {t.numel()} entries for a batch of {N}")
    if g is not None and (eps is None or alpha is None):
        raise ValueError("attack_step: a step needs eps and alpha")
    per_sample = x0.numel() // max(N, 1)
    lib = L.lib()
    nws = lib.ud_attack_workspace_bytes(N, per_sample)
    ws = L.workspace(nws, x0.device)
    L.check(lib.ud_attack_step(L.ptr(x0), L.ptr(x_adv), L.ptr(g), L.ptr(loss), L.ptr(best_loss), L.ptr(x_best),
                               L.ptr(eps), L.ptr(alpha), float(lo), float(hi), ATTACK_NORMS[norm], N, per_sample,
                               L.ptr(ws), ws.numel(), L.stream()), "attack_step")


# ------------------------------------------------------------------------------------------
# a20: image corruptions (unidefense_b200/corrupt.py)
# ------------------------------------------------------------------------------------------
CORRUPT_KINDS = {"saturation": 0, "contrast": 1, "block": 2, "noise": 3, "blur": 4, "pixelate": 5, "jpeg": 6}


def corrupt(x, kind, param, ids=None, seed=0, lo=-1.0, hi=1.0):
    """y = corruption `kind` of x at severity parameter `param` (csrc/ud_corrupt.cu; definitions in
    include/unidefense_b200.h).  x: contiguous fp32 [N, 3, H, W] in [lo, hi]; ids: int64 [N] per-sample keys of the
    random kinds (None: 0..N-1); seed: uint64.  No autograd: y has no gradient and x is not differentiated."""
    if kind not in CORRUPT_KINDS:
        raise ValueError(f"corrupt: kind must be one of {sorted(CORRUPT_KINDS)}, got {kind!r}")
    L.require_cuda_f32(x)
    if x.dim() != 4 or x.shape[1] != 3:
        raise ValueError(f"corrupt: x must be [N, 3, H, W] RGB, got {tuple(x.shape)}")
    N, _, H, W = x.shape
    if ids is not None:
        if not ids.is_cuda or ids.device != x.device or ids.dtype != torch.int64 or ids.numel() != N:
            raise ValueError(f"corrupt: ids must be an int64 tensor of {N} entries on {x.device}")
        ids = ids.contiguous()
    seed = int(seed)
    if not 0 <= seed < 2 ** 64:
        raise ValueError(f"corrupt: seed {seed} is not a uint64")
    y = torch.empty_like(x)
    lib = L.lib()
    k = CORRUPT_KINDS[kind]
    nws = lib.ud_corrupt_workspace_bytes(k, N, H, W)
    ws = L.workspace(nws, x.device) if nws else None
    L.check(lib.ud_corrupt(L.ptr(x.detach()), L.ptr(y), L.ptr(ids), N, H, W, k, float(param), seed, float(lo),
                           float(hi), L.ptr(ws), nws, L.stream()), "corrupt")
    return y
