"""a5/a6 dense projections on tcgen05 (csrc/ud_proj.cu): implicit-GEMM 1x1 / 3x3 convolution + BatchNorm partial
statistics in the epilogue, against an fp64 convolution of the same operands (oracle: F.conv2d is what
model/modules.py:82-85 / :111-114 call), the reference's DyFi fixtures, and the whole filter module."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# (N, Cin, Cout, H, W, k): EB4 freq (544 @12x7) and spat (272 @12x12); R50-style 8x8 / 8x5 (two samples per tile);
# R18-style 16x16 and 24x24 (row-block tiles); ragged channel counts (Cin % 32 != 0, Cout % 128 != 0); tiny M.
CASES = [(4, 544, 544, 12, 7, 1), (4, 272, 272, 12, 12, 3), (5, 64, 96, 8, 5, 1), (5, 64, 72, 8, 8, 3),
         (2, 128, 160, 16, 16, 3), (1, 48, 40, 24, 24, 3), (3, 36, 200, 24, 13, 1), (2, 32, 32, 3, 3, 3),
         (1, 32, 8, 1, 1, 1), (3, 100, 130, 5, 7, 3)]


def _ref(x, w):
    return F.conv2d(x.double().cpu(), w.double().cpu(), None, 1, w.shape[-1] // 2)


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_conv_and_stats(case, precision, layout):
    from unidefense_b200 import ops
    N, Cin, Cout, H, W, k = case
    g = torch.Generator().manual_seed(N * 1000 + Cin + Cout + H * 7 + W + k)
    x = torch.randn(N, Cin, H, W, generator=g) + 0.3
    w = torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5
    xd = x.cuda()
    if layout == "nhwc":
        xd = xd.contiguous(memory_format=torch.channels_last)
    y, mean, m2 = ops.proj_conv(xd, w.cuda(), precision)
    ref = _ref(x, w)
    scale = float(ref.abs().max())
    # 3xTF32: fp32-grade (the stated <=1e-4); plain TF32: 10-bit mantissa operands, the bound cuDNN's TF32 conv meets
    tol = 2e-5 if precision == "3xtf32" else 4e-3
    assert y.is_contiguous() and y.shape == ref.shape
    err = float((y.double().cpu() - ref).abs().max())
    assert err <= tol * scale, f"max abs err {err:.3e} vs scale {scale:.3e}"
    if N * H * W >= 2:
        rm = ref.mean(dim=(0, 2, 3))
        r2 = ((ref - rm[None, :, None, None]) ** 2).sum(dim=(0, 2, 3))
        stol = 1e-4 if precision == "3xtf32" else 1e-2
        torch.testing.assert_close(mean.double().cpu(), rm, rtol=stol, atol=stol * float(rm.abs().max() + ref.std()))
        torch.testing.assert_close(m2.double().cpu(), r2, rtol=stol, atol=stol * float(r2.abs().max()))


# (N, Cin, Cout, H, W, k): 1x1 -> data AND weight gradient on tcgen05; 3x3 -> data gradient on tcgen05, weight gradient
# through the library; ragged channel counts; a plane whose pixel count is not a multiple of 32 (K padding of wgrad)
GRAD_CASES = [(3, 64, 96, 8, 5, 1), (4, 544, 544, 12, 7, 1), (2, 100, 36, 6, 6, 1), (3, 64, 80, 8, 8, 3),
              (2, 272, 272, 12, 12, 3), (1, 48, 40, 24, 24, 3)]


@pytest.mark.parametrize("case", GRAD_CASES)
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
def test_gradients_match_convolution_backward(case, precision):
    from unidefense_b200 import _lib as L
    from unidefense_b200 import ops
    N, Cin, Cout, H, W, k = case
    g = torch.Generator().manual_seed(5 + Cin + Cout + k)
    x = torch.randn(N, Cin, H, W, generator=g)
    w = torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5
    gy = torch.randn(N, Cout, H, W, generator=g)
    xd, wd = x.cuda().requires_grad_(), w.cuda().requires_grad_()
    y, _, _ = ops.proj_conv(xd, wd, precision)
    before = L.lib().ud_launch_count()
    gx, gw = torch.autograd.grad((y * gy.cuda()).sum(), [xd, wd])
    launched = L.lib().ud_launch_count() - before
    assert launched >= (4 if k == 1 else 3)          # prep + tcgen05 GEMM(s) really ran in backward
    x64, w64 = x.double().requires_grad_(), w.double().requires_grad_()
    rx, rw = torch.autograd.grad((F.conv2d(x64, w64, None, 1, k // 2) * gy.double()).sum(), [x64, w64])
    tol = 3e-5 if precision == "3xtf32" else 5e-3
    assert float((gx.double().cpu() - rx).abs().max()) <= tol * float(rx.abs().max())
    assert float((gw.double().cpu() - rw).abs().max()) <= tol * float(rw.abs().max())


def test_filter_modules_use_the_tensor_core_path(golden_ops_r2):
    """FrequencyDynamicFilter / SpatialDynamicFilter (drop-in modules) against the reference fixtures with layer1[0]
    on tcgen05: forward, every gradient, running statistics."""
    import torch.nn as nn

    from unidefense_b200 import _lib as L
    from unidefense_b200 import ops
    from unidefense_b200.model import modules as M
    for c in golden_ops_r2["dyfi_wide"]:
        depth = c["x"].shape[1] // (2 if c["kind"] == "freq" else 1)
        act = M.MemoryEfficientSwish if c["act"] == "swish" else nn.ReLU
        cls = M.FrequencyDynamicFilter if c["kind"] == "freq" else M.SpatialDynamicFilter
        mod = cls(depth, act, nn.BatchNorm2d, True, False).cuda().train()
        mod.load_state_dict(c["sd0"])
        x = c["x"].cuda().requires_grad_()
        assert ops.proj_supported(x, mod.layer1[0])             # the module selects the tcgen05 projection
        before = L.lib().ud_launch_count()
        out = mod(x, c["diff"].cuda())
        assert x.shape[1] >= 32 and x.shape[1] % 4 == 0
        assert L.lib().ud_launch_count() - before >= 5          # prep x, prep w, gemm, merge + the mask stage
        scale_m, scale_o = float(c["mask"].abs().max()), float(c["out"].abs().max())
        torch.testing.assert_close(out["mask"].cpu(), c["mask"], rtol=1e-4, atol=1e-5 * scale_m)
        torch.testing.assert_close(out["out"].cpu(), c["out"], rtol=1e-4, atol=1e-5 * scale_o)
        ps = [mod.layer1[0].weight, mod.layer1[1].weight, mod.layer1[1].bias, mod.layer2[0].weight]
        gs = torch.autograd.grad((out["mask"] * c["gm"].cuda()).sum() + (out["out"] * c["go"].cuda()).sum(), [x] + ps)
        for a, k in zip(gs, ["gx", "gw1", "ggamma", "gbeta", "gw2"]):
            torch.testing.assert_close(a.cpu(), c[k], rtol=2e-4, atol=2e-5 * float(c[k].abs().max()) + 1e-7)
        sd = mod.state_dict()
        for k in ("layer1.1.running_mean", "layer1.1.running_var"):
            torch.testing.assert_close(sd[k].cpu(), c["sd1"][k], rtol=1e-4, atol=1e-6)


def test_unsupported_shapes_are_reported():
    from unidefense_b200 import _lib as L
    lib = L.lib()
    rc = lib.ud_proj_fwd(None, None, None, None, None, None, None, None, 2, 4, 4, 6, 8, 1, None)
    assert rc < 0 and b"multiple of 4" in lib.ud_last_error()
    rc = lib.ud_proj_fwd(None, None, None, None, None, None, None, None, 2, 4, 4, 64, 8, 5, None)
    assert rc < 0 and b"kernel size" in lib.ud_last_error()
