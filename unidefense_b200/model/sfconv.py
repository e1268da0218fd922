"""Spatial-frequency convolutions of the backbones (stock torch; SURVEY.md §8a row a17, scope "next").

Reference: SFConv2dStaticSamePadding (model/efficientnet/exp.py:7-65) and SFConv2d
(model/resnet/exp.py:21-54).  Both are an nn.Conv2d (the spatial branch, so the pretrained
`weight` key loads unchanged) that owns a second dense 1x1 convolution `freq_conv` on the
cat([re, im]) half spectrum and a scalar gate `sf_coef` (init -10):

    y = (1 - sigmoid(sf_coef)) * conv(x) + sigmoid(sf_coef) * pool(irfft2(freq_conv(cat rfft2(x))))

The north star keeps the backbone on stock torch, so this file is plain PyTorch; the FFTs are
computed in fp32 even under bf16 autocast (torch.complex rejects bf16, SURVEY.md §0).
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F


# Under bf16 autocast with channels-last activations (the benchmark configuration) the two small 2-D transforms are
# evaluated as DFT-by-GEMM on the tensor cores: with x stored [N, h, w, C], rfft2 + cat([re, im]) is
#     V = L @ x.view(N, h, w*C)            L [2h x h]   rows (j, ri):  cos / -sin of 2 pi j r / h
#     P = R @ V.view(N*h, 2w, C)           R [2wh x 2w] rows (k, ri'), cols (ri, s): complex product with e^{-2 pi i k s / w}
# and P viewed [N, h, wh, 2C] IS the channels-last planar spectrum the 1x1 convolution consumes; the inverse
# (tensor_split + complex + irfft2, c2r semantics) is
#     G = Li @ Q.view(N, h, wh*2C)         Li [2h x h]  rows (r, p): cos / sin of 2 pi j r / h
#     y = A  @ G.view(N*h, 4wh, C)         A [w x 4wh]  folds the complex product and the Hermitian weights m_k
# Four batched library GEMMs replace copy->fp32, R2C, C2C, pack, unpack, C2R and their backward twins; autograd
# differentiates the matmuls.  Exact fp32 runs keep the cuFFT path (bf16 twiddles carry ~3 significant digits).
# largest side evaluated as DFT-by-GEMM: 96 covers every SFConv layer of the shipped configs (95^2 at EB4@380 is the
# biggest: with it on the GEMM path the step went 77.2 -> 74.0 ms on a B200; 64 was the round-1 setting)
_DFT_MAX = 96
_dft_cache = {}


def _dft_mats(h, w, norm, device):
    key = (h, w, norm, str(device))
    if key in _dft_cache:
        return _dft_cache[key]
    wh = w // 2 + 1
    dd = torch.float64
    fs = 1.0 / math.sqrt(h * w) if norm == "ortho" else 1.0            # forward scale
    is_ = 1.0 / math.sqrt(h * w) if norm == "ortho" else 1.0 / (h * w)  # inverse scale
    ah = 2 * math.pi * torch.outer(torch.arange(h, dtype=dd), torch.arange(h, dtype=dd)) / h      # [j, r]
    aw = 2 * math.pi * torch.outer(torch.arange(wh, dtype=dd), torch.arange(w, dtype=dd)) / w     # [k, s]
    ch, sh, cw, sw = torch.cos(ah), torch.sin(ah), torch.cos(aw), torch.sin(aw)
    # forward, height: V[(j, ri), r]
    L = torch.stack([ch, -sh], dim=1).reshape(2 * h, h)
    # forward, width: P[(k, ri'), (ri, s)] : re' = cw*re + sw*im ; im' = -sw*re + cw*im
    R = torch.stack([torch.cat([cw, sw], dim=1), torch.cat([-sw, cw], dim=1)], dim=1).reshape(2 * wh, 2 * w) * fs
    # inverse, height: G[(r, p), j] : p=0 -> cos, p=1 -> sin   (e^{+i})
    Li = torch.stack([ch.t(), sh.t()], dim=1).reshape(2 * h, h)
    # inverse, width: y[s] = sum_k m_k (Tre cos - Tim sin), Tre = G0[ri0] - G1[ri1], Tim = G1[ri0] + G0[ri1]
    m = torch.full((wh,), 2.0, dtype=dd)
    m[0] = 1.0
    if w % 2 == 0:
        m[-1] = 1.0
    cm, sm = (cw * m[:, None]).t(), (sw * m[:, None]).t()          # [s, k]
    a0 = torch.stack([cm, -sm], dim=2).reshape(w, 2 * wh)          # cols (k, ri) acting on G0
    a1 = torch.stack([-sm, -cm], dim=2).reshape(w, 2 * wh)         # cols (k, ri) acting on G1
    A = torch.cat([a0, a1], dim=1) * is_                           # [w, (p, k, ri)]
    mats = tuple(t.to(device=device, dtype=torch.float32) for t in (L, R, Li, A))
    _dft_cache[key] = mats
    return mats


def _dft_gemm_ok(x):
    h, w = x.shape[-2:]
    # bf16 autocast only: under fp16 autocast (or none) the transforms stay on the fp32 cuFFT path (ADVICE r1)
    return (x.is_cuda and torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.bfloat16
            and x.dim() == 4 and h <= _DFT_MAX and w <= _DFT_MAX
            and x.is_contiguous(memory_format=torch.channels_last) and not x.is_contiguous())


def _sf_forward_gemm(x, spat, freq_conv, sf_coef, norm):
    N, C, h, w = x.shape
    wh = w // 2 + 1
    L, R, Li, A = _dft_mats(h, w, norm, x.device)
    xl = x.permute(0, 2, 3, 1)                                        # [N, h, w, C] view of the channels-last storage
    V = torch.matmul(L, xl.reshape(N, h, w * C))                      # [N, 2h, w*C]  = [n, j, ri, s, c]
    P = torch.matmul(R, V.reshape(N * h, 2 * w, C))                   # [N*h, 2wh, C] = [n, j, k, ri', c]
    planar = P.reshape(N, h, wh, 2 * C).permute(0, 3, 1, 2)           # channels-last [N, 2C, h, wh]
    Q = freq_conv(planar)
    Co = Q.shape[1] // 2
    Ql = Q.permute(0, 2, 3, 1).reshape(N, h, wh * 2 * Co)             # [n, j, (k, ri, c)]
    G = torch.matmul(Li, Ql)                                          # [N, 2h, ...]  = [n, r, p, k, ri, c]
    y = torch.matmul(A, G.reshape(N * h, 4 * wh, Co))                 # [N*h, w, Co]
    y = y.reshape(N, h, w, Co).permute(0, 3, 1, 2)                    # channels-last [N, Co, h, w]
    if tuple(y.shape[-2:]) != tuple(spat.shape[-2:]):
        y = F.adaptive_avg_pool2d(y, spat.shape[-2:])
    return torch.lerp(spat, y.to(spat.dtype), torch.sigmoid(sf_coef).to(spat.dtype))


# SURVEY.md §8(f) #1, first step: on CUDA the ~10 elementwise / layout / dtype passes torch makes around the two
# FFTs and the 1x1 convolution (x.float, real, imag, cat, cast, tensor_split, complex, two muls, add and their
# backward twins) are replaced by three single-pass kernels (ops.sf_pack / sf_unpack / sf_mix); cuFFT and the
# convolution stay library calls.
def _sf_forward_glue(x, spat, freq_conv, sf_coef, norm):
    from .. import ops
    size = x.shape[-2:]
    xf = x.to(dtype=torch.float32, memory_format=torch.contiguous_format)
    with torch.autocast(device_type="cuda", enabled=False):
        spec = torch.fft.rfft2(xf, norm=norm)
    cl = spat.dim() == 4 and spat.is_contiguous(memory_format=torch.channels_last) and not spat.is_contiguous()
    planar = ops.sf_pack(spec, spat.dtype if spat.dtype in (torch.float32, torch.bfloat16) else torch.float32, cl)
    planar = freq_conv(planar)
    with torch.autocast(device_type="cuda", enabled=False):
        y = torch.fft.irfft2(ops.sf_unpack(planar), s=size, norm=norm)
    if tuple(y.shape[-2:]) != tuple(spat.shape[-2:]):
        y = F.adaptive_avg_pool2d(y, spat.shape[-2:])
    return ops.sf_mix(spat, y, sf_coef)


# The plain torch composition of the reference: the CPU path (the oracle arm).
def _sf_forward_plain(x, spat, freq_conv, sf_coef, norm):
    size = x.shape[-2:]
    with torch.autocast(device_type=x.device.type, enabled=False):
        spec = torch.fft.rfft2(x.float(), norm=norm)
        planar = torch.cat([spec.real, spec.imag], dim=1)
    planar = freq_conv(planar)
    with torch.autocast(device_type=x.device.type, enabled=False):
        re, im = torch.tensor_split(planar.float(), 2, dim=1)
        y = torch.fft.irfft2(torch.complex(re, im), s=size, norm=norm)
    if tuple(y.shape[-2:]) != tuple(spat.shape[-2:]):
        y = F.adaptive_avg_pool2d(y, spat.shape[-2:])
    gate = torch.sigmoid(sf_coef)
    return (1.0 - gate) * spat + gate * y


def _sf_forward(x, spat, freq_conv, sf_coef, norm):
    """(1 - sigmoid(sf_coef)) * spat + sigmoid(sf_coef) * pool(irfft2(freq_conv(cat rfft2(x))))."""
    if _dft_gemm_ok(x):
        return _sf_forward_gemm(x, spat, freq_conv, sf_coef, norm)
    if x.is_cuda:
        return _sf_forward_glue(x, spat, freq_conv, sf_coef, norm)
    return _sf_forward_plain(x, spat, freq_conv, sf_coef, norm)


class SFConv2d(nn.Conv2d):
    """model/resnet/exp.py:21-54."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, freq_norm=None, **kwargs):
        super().__init__(in_channels, out_channels, kernel_size, stride, **kwargs)
        self.freq_norm = freq_norm
        self.freq_conv = nn.Conv2d(in_channels * 2, out_channels * 2, kernel_size=1, bias=False)
        self.sf_coef = nn.Parameter(torch.tensor(-10.0))

    def forward(self, x):
        spat = self._conv_forward(x, self.weight, self.bias)
        return _sf_forward(x, spat, self.freq_conv, self.sf_coef, self.freq_norm)


def same_pad_amounts(size, kernel, stride, dilation=1):
    """TensorFlow 'SAME' padding for a nominal input extent -> (before, after)."""
    out = math.ceil(size / stride)
    total = max((out - 1) * stride + (kernel - 1) * dilation + 1 - size, 0)
    return total // 2, total - total // 2


class SamePadConv2d(nn.Conv2d):
    """Conv2d with static TF-'SAME' padding computed from the nominal image size at construction
    (model/efficientnet/utils.py Conv2dStaticSamePadding); keeps a parameter-free `static_padding`
    child like the reference so module trees line up."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, image_size=None, **kwargs):
        super().__init__(in_channels, out_channels, kernel_size, stride, **kwargs)
        ih, iw = (image_size, image_size) if isinstance(image_size, int) else image_size
        top, bottom = same_pad_amounts(ih, self.kernel_size[0], self.stride[0], self.dilation[0])
        left, right = same_pad_amounts(iw, self.kernel_size[1], self.stride[1], self.dilation[1])
        self.static_padding = nn.ZeroPad2d((left, right, top, bottom)) if (top + bottom + left + right) else nn.Identity()

    def forward(self, x):
        return self._conv_forward(self.static_padding(x), self.weight, self.bias)


class SFSamePadConv2d(SamePadConv2d):
    """model/efficientnet/exp.py:7-65."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, image_size=None, freq_norm=None, **kwargs):
        super().__init__(in_channels, out_channels, kernel_size, stride, image_size=image_size, **kwargs)
        self.freq_norm = freq_norm
        self.freq_conv = nn.Conv2d(in_channels * 2, out_channels * 2, kernel_size=1, bias=False)
        self.sf_coef = nn.Parameter(torch.tensor(-10.0))

    def forward(self, x):
        spat = self._conv_forward(self.static_padding(x), self.weight, self.bias)
        return _sf_forward(x, spat, self.freq_conv, self.sf_coef, self.freq_norm)
