"""a17 (next row): SFConv modules (stock torch FFT/conv + our pack / unpack / mix glue kernels) vs the reference
fixtures, and the glue kernels vs their torch compositions in every dtype / memory-format combination."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def close(a, b, rtol=1e-4, atol=None):
    b = b.detach()
    scale = float(b.abs().max()) if b.numel() else 1.0
    atol = (1e-5 * max(scale, 1e-6)) if atol is None else atol
    torch.testing.assert_close(a.detach().float().cpu(), b.float().cpu(), rtol=rtol, atol=atol)


@pytest.mark.parametrize("shape", [(2, 6, 5, 3), (3, 64, 12, 7), (2, 130, 24, 13), (1, 7, 4, 3), (2, 336, 48, 25)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("cl", [False, True])
def test_pack_unpack(shape, dtype, cl):
    from unidefense_b200 import ops
    N, C, h, wh = shape
    g = torch.Generator().manual_seed(C)
    spec = torch.complex(torch.randn(shape, generator=g), torch.randn(shape, generator=g)).cuda().requires_grad_()
    planar = ops.sf_pack(spec, dtype, cl)
    want = torch.cat([spec.real, spec.imag], dim=1).to(dtype)
    assert planar.shape == want.shape and planar.dtype == dtype
    if cl and C % 2 == 0:
        assert planar.is_contiguous(memory_format=torch.channels_last)
    torch.testing.assert_close(planar.float(), want.float(), rtol=0, atol=0)
    w = torch.randn(want.shape, generator=g).cuda()
    (planar.float() * w).sum().backward()
    gw = torch.complex(*torch.tensor_split(w.to(dtype).float() if False else w, 2, dim=1))
    tol = 1e-2 if dtype == torch.bfloat16 else 1e-6
    torch.testing.assert_close(torch.view_as_real(spec.grad), torch.view_as_real(gw), rtol=tol, atol=tol)
    # unpack is the inverse (and pack's adjoint)
    p2 = planar.detach().clone().requires_grad_()
    back = ops.sf_unpack(p2)
    torch.testing.assert_close(torch.view_as_real(back), torch.view_as_real(torch.complex(*torch.tensor_split(p2.detach().float(), 2, dim=1))))
    gz = torch.complex(torch.randn(shape, generator=g), torch.randn(shape, generator=g)).cuda()
    torch.view_as_real(back).mul(torch.view_as_real(gz)).sum().backward()
    torch.testing.assert_close(p2.grad.float(), torch.cat([gz.real, gz.imag], 1).to(dtype).float(), rtol=0, atol=0)


@pytest.mark.parametrize("shape", [(2, 6, 5, 5), (3, 64, 12, 12), (2, 130, 7, 9), (1, 7, 4, 4), (2, 336, 24, 24)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("cl", [False, True])
def test_mix(shape, dtype, cl):
    from unidefense_b200 import ops
    g = torch.Generator().manual_seed(shape[1])
    spat = torch.randn(shape, generator=g).to(dtype).cuda()
    if cl:
        spat = spat.contiguous(memory_format=torch.channels_last)
    freq = torch.randn(shape, generator=g).cuda()
    coef = torch.tensor(0.3).cuda()
    gout = torch.randn(shape, generator=g).cuda()
    leaves = [spat.clone().requires_grad_(), freq.clone().requires_grad_(), coef.clone().requires_grad_()]
    out = ops.sf_mix(*leaves)
    assert out.dtype == dtype and out.shape == spat.shape
    (out.float() * gout).sum().backward()
    ref = [spat.double().requires_grad_(), freq.double().requires_grad_(), coef.double().requires_grad_()]
    s = torch.sigmoid(ref[2])
    o64 = (1 - s) * ref[0] + s * ref[1]
    (o64 * gout.double()).sum().backward()
    tol = 2e-2 if dtype == torch.bfloat16 else 1e-5
    close(out, o64, rtol=tol, atol=tol)
    close(leaves[0].grad, ref[0].grad, rtol=tol, atol=tol)
    close(leaves[1].grad, ref[1].grad, rtol=tol, atol=tol)
    close(leaves[2].grad, ref[2].grad, rtol=2e-2 if dtype == torch.bfloat16 else 1e-3,
          atol=(2e-2 if dtype == torch.bfloat16 else 1e-4) * float(ref[2].grad.abs()) + 1e-4)


@pytest.mark.parametrize("cl", [False, True])
def test_sfconv_modules_reference_fixture(golden_ops, cl):
    from unidefense_b200.model.sfconv import SFConv2d, SFSamePadConv2d
    for c in golden_ops["sfconv"]:
        C, hw, s = c["x"].shape[1], c["x"].shape[-1], c["stride"]
        if c["kind"] == "eff":
            m = SFSamePadConv2d(C, C, 3, stride=s, image_size=hw, freq_norm=c["norm"], groups=C, bias=False)
        else:
            m = SFConv2d(C, C, 3, stride=s, padding=1, bias=False, freq_norm=c["norm"])
        m.load_state_dict(c["sd"])
        m = m.cuda()
        x = c["x"].cuda()
        if cl:
            m = m.to(memory_format=torch.channels_last)
            x = x.contiguous(memory_format=torch.channels_last)
        x.requires_grad_()
        y = m(x)
        close(y, c["y"], rtol=1e-4, atol=2e-5)
        (y * c["gy"].cuda()).sum().backward()
        close(x.grad, c["gx"], rtol=1e-3, atol=1e-4 * float(c["gx"].abs().max()))
        close(m.freq_conv.weight.grad, c["gfw"], rtol=1e-3, atol=1e-4 * float(c["gfw"].abs().max()))
        assert m.sf_coef.grad is not None and m.weight.grad is not None


@pytest.mark.parametrize("cfg", [(48, 24, 5, 2), (32, 12, 3, 1), (16, 48, 3, 1), (24, 95, 5, 2), (8, 96, 3, 1)])
def test_sfconv_paths_agree_bf16(cfg):
    """bf16 autocast + channels_last (the bench configuration): DFT-by-GEMM path and glue-kernel path vs the plain
    torch composition (bf16 tolerance: the twiddles themselves are bf16 in the GEMM path)."""
    from unidefense_b200.model import sfconv
    C, hw, k, stride = cfg
    torch.manual_seed(0)
    m = sfconv.SFSamePadConv2d(C, C, k, stride=stride, image_size=hw, freq_norm="ortho", groups=C, bias=False).cuda()
    with torch.no_grad():
        m.sf_coef.fill_(0.2)
    m = m.to(memory_format=torch.channels_last)
    x = torch.randn(4, C, hw, hw, device="cuda").contiguous(memory_format=torch.channels_last)
    outs = {}
    paths = {"gemm": sfconv._sf_forward_gemm, "glue": sfconv._sf_forward_glue, "plain": sfconv._sf_forward_plain}
    for mode, sf_forward in paths.items():
        xi = x.clone().requires_grad_()
        m.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            assert sfconv._dft_gemm_ok(xi)          # the module itself takes the GEMM path here
            spat = m._conv_forward(m.static_padding(xi), m.weight, m.bias)
            y = sf_forward(xi, spat, m.freq_conv, m.sf_coef, m.freq_norm)
        y.float().square().mean().backward()
        outs[mode] = (y.float(), xi.grad.float(), m.freq_conv.weight.grad.clone(), m.sf_coef.grad.clone().reshape(1),
                      m.weight.grad.clone())
    for mode in ("gemm", "glue"):
        for a, b in zip(outs[mode], outs["plain"]):
            torch.testing.assert_close(a, b, rtol=5e-2, atol=3e-2 * float(b.abs().max()) + 1e-6)


def test_dft_gemm_matrices_fp32():
    """The four DFT matrices reproduce rfft2+cat and tensor_split+complex+irfft2 exactly when run in fp32."""
    from unidefense_b200.model import sfconv
    for (h, w) in [(12, 12), (24, 24), (48, 48), (9, 7), (8, 6), (95, 95), (96, 64)]:
        for norm in ("ortho", None):
            N, C = 2, 6
            wh = w // 2 + 1
            L, R, Li, A = sfconv._dft_mats(h, w, norm, torch.device("cuda"))
            x = torch.randn(N, C, h, w, device="cuda").contiguous(memory_format=torch.channels_last)
            V = torch.matmul(L, x.permute(0, 2, 3, 1).reshape(N, h, w * C))
            planar = torch.matmul(R, V.reshape(N * h, 2 * w, C)).reshape(N, h, wh, 2 * C).permute(0, 3, 1, 2)
            f = torch.fft.rfft2(x, norm=norm)
            want = torch.cat([f.real, f.imag], 1)
            torch.testing.assert_close(planar, want, rtol=1e-4, atol=1e-5 * float(want.abs().max()))
            Q = torch.randn(N, 2 * C, h, wh, device="cuda").contiguous(memory_format=torch.channels_last)
            G = torch.matmul(Li, Q.permute(0, 2, 3, 1).reshape(N, h, wh * 2 * C))
            y = torch.matmul(A, G.reshape(N * h, 4 * wh, C)).reshape(N, h, w, C).permute(0, 3, 1, 2)
            re, im = torch.tensor_split(Q, 2, dim=1)
            want = torch.fft.irfft2(torch.complex(re.contiguous(), im.contiguous()), s=(h, w), norm=norm)
            torch.testing.assert_close(y, want, rtol=1e-4, atol=1e-5 * float(want.abs().max()))
