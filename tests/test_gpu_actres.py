"""Residuals stored leaky_relu'd: hg_conv1d_fwd_actres and hg_resblock_pair_fwd_actin rebuild the raw residual
r = min(a, a / slope) from its activated bf16 copy `a` in the epilogue (the Generator forward keeps one copy of a
tensor that feeds both a conv and a residual add)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SLOPE = 0.1


@pytest.fixture(scope="module")
def L():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from hifigan_b200 import _lib
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return _lib.lib()


def _unact(a):
    """the residual the kernels rebuild from its activated copy, in fp32"""
    a = a.float()
    return torch.where(a < 0, a * (1.0 / SLOPE), a)


def _pack(L, w, k, c_in, c_out):
    from hifigan_b200 import _lib
    wp = torch.empty(k, c_out, c_in, dtype=torch.bfloat16, device="cuda")
    _lib.check(L.hg_pack_conv1d_weight(w.data_ptr(), 0, c_out, c_in, k, c_in, wp.data_ptr(),
                                       torch.cuda.current_stream().cuda_stream))
    return wp


@pytest.mark.parametrize("b,t,cin,cout,k,d", [(2, 300, 64, 64, 11, 5), (2, 1000, 128, 128, 3, 1),
                                              (4, 8192, 256, 256, 3, 1), (2, 257, 32, 32, 7, 3)])
@pytest.mark.parametrize("mrf", [False, True])
def test_conv1d_fwd_actres_vs_torch_fp32(L, b, t, cin, cout, k, d, mrf):
    """forward flavours 0 (one residual) and 5 (MRF-final: two more addends, scale) on the plain and the CTA-pair
    kernel; tolerance as test_gpu_parity.test_conv1d_fwd_vs_torch_fp32"""
    from hifigan_b200 import _lib
    g = torch.Generator().manual_seed(b * t + cout + k + mrf)
    x = torch.randn(b, t, cin, generator=g).cuda().bfloat16()
    w = (torch.randn(cout, cin, k, generator=g) / (cin * k) ** 0.5).cuda()
    bias = torch.randn(cout, generator=g).cuda()
    r0 = F.leaky_relu(torch.randn(b, t, cout, generator=g).cuda(), SLOPE).bfloat16()
    r1, r2 = (torch.randn(b, t, cout, generator=g).cuda().bfloat16() for _ in range(2))
    wp = _pack(L, w, k, cin, cout)
    out_raw = torch.full((b, t, cout), 7.0, dtype=torch.bfloat16, device="cuda")
    out_act = torch.full((b, t, cout), 7.0, dtype=torch.bfloat16, device="cuda")
    scale = 1.0 / 3 if mrf else 1.0
    pad = (k - 1) * d // 2
    _lib.check(L.hg_conv1d_fwd_actres(x.data_ptr(), wp.data_ptr(), bias.data_ptr(), b, t, cin, cout, k, d, pad,
                                      r0.data_ptr(), SLOPE, r1.data_ptr() if mrf else 0, r2.data_ptr() if mrf else 0,
                                      scale, out_raw.data_ptr(), out_act.data_ptr(), SLOPE, 0, 1,
                                      torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = F.conv1d(x.float().transpose(1, 2), wp.float().permute(1, 2, 0).contiguous(), bias, dilation=d,
                   padding=pad).transpose(1, 2) + _unact(r0)
    if mrf:
        ref = (ref + r1.float() + r2.float()) * scale
    tol = 2.0 ** -8 * ref.abs() + 1e-3
    assert bool(((out_raw.float() - ref).abs() <= tol).all())
    assert bool(((out_act.float() - F.leaky_relu(ref, SLOPE)).abs() <= tol).all())


def test_conv1d_fwd_actres_slope_one_is_the_raw_residual(L):
    """res0_slope = 1: the residual is taken as it is, bit for bit what hg_conv1d_fwd computes"""
    from hifigan_b200 import _lib
    b, t, c, k = 2, 600, 64, 3
    g = torch.Generator().manual_seed(5)
    x = torch.randn(b, t, c, generator=g).cuda().bfloat16()
    wp = _pack(L, (torch.randn(c, c, k, generator=g) / (c * k) ** 0.5).cuda(), k, c, c)
    bias = torch.randn(c, generator=g).cuda()
    r0 = torch.randn(b, t, c, generator=g).cuda().bfloat16()
    st = torch.cuda.current_stream().cuda_stream
    outs = [torch.empty(b, t, c, dtype=torch.bfloat16, device="cuda") for _ in range(2)]
    _lib.check(L.hg_conv1d_fwd(x.data_ptr(), wp.data_ptr(), bias.data_ptr(), b, t, c, c, k, 1, 1, r0.data_ptr(), 0,
                               0, 1.0, outs[0].data_ptr(), 0, SLOPE, 0, 1, st))
    _lib.check(L.hg_conv1d_fwd_actres(x.data_ptr(), wp.data_ptr(), bias.data_ptr(), b, t, c, c, k, 1, 1,
                                      r0.data_ptr(), 1.0, 0, 0, 1.0, outs[1].data_ptr(), 0, SLOPE, 0, 1, st))
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    for bad in (0.0, -0.1, 2.0):
        assert L.hg_conv1d_fwd_actres(x.data_ptr(), wp.data_ptr(), bias.data_ptr(), b, t, c, c, k, 1, 1,
                                      r0.data_ptr(), bad, 0, 0, 1.0, outs[1].data_ptr(), 0, SLOPE, 0, 1, st) != 0
        assert b"slope" in L.hg_last_error()


@pytest.mark.parametrize("c,k,d,two", [(64, 3, 1, True), (64, 7, 5, True), (32, 11, 5, True), (64, 5, 6, False),
                                       (32, 3, 2, False)])
@pytest.mark.parametrize("mrf", [False, True])
def test_resblock_pair_fwd_actin_vs_torch_fp32(L, c, k, d, two, mrf):
    """the fused ResBlock1 step (two=True) and ResBlock2 step on x_act = bf16(leaky_relu(x)): the kernel skips its
    own first leaky_relu and rebuilds the residual; plain instantiation and the general one (mrf: addends, scale,
    activated output).  Tolerances as the raw-input tests in test_gpu_parity."""
    from hifigan_b200 import _lib
    b, t = 2, 700
    g = torch.Generator().manual_seed(c * 1000 + k * 10 + d + mrf)
    xa = F.leaky_relu(torch.randn(b, t, c, generator=g).cuda(), SLOPE).bfloat16()
    w1 = (torch.randn(c, c, k, generator=g) / (c * k) ** 0.5).cuda()
    w2 = (torch.randn(c, c, k, generator=g) / (c * k) ** 0.5).cuda()
    b1, b2 = torch.randn(c, generator=g).cuda(), torch.randn(c, generator=g).cuda()
    r1, r2 = (torch.randn(b, t, c, generator=g).cuda().bfloat16() for _ in range(2))
    wp1 = _pack(L, w1, k, c, c)
    wp2 = _pack(L, w2, k, c, c) if two else None
    out_raw = torch.full((b, t, c), 7.0, dtype=torch.bfloat16, device="cuda")
    out_act = torch.full((b, t, c), 7.0, dtype=torch.bfloat16, device="cuda")
    scale = 1.0 / 3 if mrf else 1.0
    _lib.check(L.hg_resblock_pair_fwd_actin(xa.data_ptr(), wp1.data_ptr(), b1.data_ptr(),
                                            wp2.data_ptr() if two else 0, b2.data_ptr() if two else 0, b, t, c, k, d,
                                            SLOPE, r1.data_ptr() if mrf else 0, r2.data_ptr() if mrf else 0, scale,
                                            out_raw.data_ptr(), out_act.data_ptr() if mrf else 0, 0.01, 0, 1,
                                            torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    y = F.conv1d(xa.float().transpose(1, 2), wp1.float().permute(1, 2, 0).contiguous(), b1, dilation=d,
                 padding=(k - 1) * d // 2)
    if two:
        t1 = F.leaky_relu(y, SLOPE).bfloat16().float()
        y = F.conv1d(t1, wp2.float().permute(1, 2, 0).contiguous(), b2, padding=(k - 1) // 2)
    ref = y.transpose(1, 2) + _unact(xa)
    if mrf:
        ref = (ref + r1.float() + r2.float()) * scale
    tol = 2.0 ** -8 * ref.abs() + (1.5e-2 if two else 2e-3)
    assert bool(((out_raw.float() - ref).abs() <= tol).all())
    if mrf:
        assert bool(((out_act.float() - F.leaky_relu(ref, 0.01)).abs() <= tol).all())
