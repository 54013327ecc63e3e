"""One small invocation per kernel family, for compute-sanitizer (SURVEY §5 "race detection / sanitizers"; VERDICT r1
missing item 5).  Tool, not a pytest module.

    compute-sanitizer --tool memcheck  python tests/sanitize_cases.py [family ...]
    compute-sanitizer --tool racecheck python tests/sanitize_cases.py conv pair mel
    compute-sanitizer --tool synccheck python tests/sanitize_cases.py ...

Families: conv (conv1d_tc_kernel, resident + ring weights, strided / grouped), conv2 (conv1d_tc2_kernel, CTA pairs),
pair (resblock_pair_kernel, C = 32 / 64, one- and two-conv steps), wgrad (wgrad_tc_kernel wide / narrow / grouped),
mel (mel_kernel2, mel_dft_kernel, mel_bwd_kernel), ends (the Cin = 1 / Cout = 1 discriminator kernels, pooling, packs),
step (one whole TrainStep at batch 1: every kernel of the training path, lanes included).
Each case also checks its result against torch so a sanitizer-clean but wrong kernel cannot pass.  Shapes are the
smallest that still exercise every code path (ring wrap-around, several tiles per CTA, partial last tile).
"""
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hifigan_b200 as H                     # noqa: E402
from hifigan_b200 import _lib                # noqa: E402

L = _lib.lib()
dev = torch.device("cuda")


def st():
    return torch.cuda.current_stream().cuda_stream


# compute-sanitizer is closed on this GPU pool (profiles/r02_sanitizer_closed.txt), so every output of the cases below
# is allocated between two guard bands filled with a sentinel bit pattern; check_guards() fails if any kernel wrote
# outside its tensor.  (Out-of-bounds READS are caught indirectly: inputs sit in guarded NaN-filled buffers too, and a
# stray read of a NaN poisons a result that is compared with torch.)
_GUARD = 4096          # bytes on either side
_guards = []


def guarded(shape, dtype, fill=None):
    n = 1
    for d in shape:
        n *= d
    esz = torch.empty((), dtype=dtype).element_size()
    raw = torch.full((n * esz + 2 * _GUARD,), 0xA5, dtype=torch.uint8, device=dev)
    t = raw[_GUARD:_GUARD + n * esz].view(dtype).view(*shape)
    if fill is not None:
        t.copy_(fill.to(dev).to(dtype).reshape(shape))
    _guards.append(raw)
    return t


def check_guards(what):
    torch.cuda.synchronize()
    for raw in _guards:
        lo, hi = raw[:_GUARD], raw[-_GUARD:]
        assert bool((lo == 0xA5).all()) and bool((hi == 0xA5).all()), f"{what}: a kernel wrote outside its output tensor"
    _guards.clear()


def _conv_case(b, t, cin, cout, k, d):
    g = torch.Generator().manual_seed(k * 131 + cin)
    pad = (k - 1) * d // 2
    w = (torch.randn(cout, cin, k, generator=g) / (cin * k) ** 0.5).to(dev)
    wp = torch.empty(k, cout, cin, dtype=torch.bfloat16, device=dev)
    _lib.check(L.hg_pack_conv1d_weight(w.data_ptr(), 0, cout, cin, k, cin, wp.data_ptr(), st()))
    bias = torch.randn(cout, generator=g).to(dev)
    x = guarded((b, t, cin), torch.bfloat16, torch.randn(b, t, cin, generator=g))
    res = guarded((b, t, cout), torch.bfloat16, torch.randn(b, t, cout, generator=g))
    out_r = guarded((b, t, cout), torch.bfloat16)
    out_a = guarded((b, t, cout), torch.bfloat16)
    _lib.check(L.hg_conv1d_fwd(x.data_ptr(), wp.data_ptr(), bias.data_ptr(), b, t, cin, cout, k, d, pad, res.data_ptr(),
                               0, 0, 1.0, out_r.data_ptr(), out_a.data_ptr(), 0.1, 0, 1, st()), "hg_conv1d_fwd")
    check_guards(f"conv {cin}->{cout} k{k} d{d}")
    ref = F.conv1d(x.float().transpose(1, 2), wp.float().permute(1, 2, 0).contiguous(), bias, dilation=d,
                   padding=pad).transpose(1, 2) + res.float()
    assert bool(((out_r.float() - ref).abs() <= 2.0 ** -7 * ref.abs() + 2e-3).all()), (cin, cout, k, d)
    assert bool(((out_a.float() - F.leaky_relu(ref, 0.1)).abs() <= 2.0 ** -7 * ref.abs() + 2e-3).all())


def conv():
    _conv_case(2, 300, 64, 64, 3, 1)       # resident weights, SW128
    _conv_case(2, 333, 32, 32, 7, 3)       # resident, SW64, partial tile
    _conv_case(1, 260, 256, 256, 11, 5)    # weight ring, several K chunks, ring wrap-around (below the pair threshold)
    _conv_case(160, 129, 128, 128, 3, 1)   # more tiles than SMs: persistent loop, double-buffered accumulators
    print("conv ok", flush=True)


def conv2():
    _conv_case(40, 512, 256, 256, 7, 3)    # 160 tiles >= 148: CTA-pair kernel (cta_group::2), N = 256
    _conv_case(75, 260, 128, 128, 11, 1)   # N = 128 pairs, odd tile count per item (one CTA of a pair idles)
    print("conv2 ok", flush=True)


def pair():
    for c, k, d in ((32, 3, 1), (32, 11, 5), (64, 3, 3), (64, 7, 1)):
        if not L.hg_resblock_pair_supported(c, k, d):
            continue
        g = torch.Generator().manual_seed(c + k)
        b, t = 3, 700
        mk = lambda: (torch.randn(c, c, k, generator=g) / (c * k) ** 0.5).to(dev)
        w1, w2 = mk(), mk()
        p1 = torch.empty(k, c, c, dtype=torch.bfloat16, device=dev)
        p2 = torch.empty_like(p1)
        _lib.check(L.hg_pack_conv1d_weight(w1.data_ptr(), 0, c, c, k, c, p1.data_ptr(), st()))
        _lib.check(L.hg_pack_conv1d_weight(w2.data_ptr(), 0, c, c, k, c, p2.data_ptr(), st()))
        b1, b2 = torch.randn(c, generator=g).to(dev), torch.randn(c, generator=g).to(dev)
        x = guarded((b, t, c), torch.bfloat16, torch.randn(b, t, c, generator=g))
        out = guarded((b, t, c), torch.bfloat16)
        _lib.check(L.hg_resblock_pair_fwd(x.data_ptr(), p1.data_ptr(), b1.data_ptr(), p2.data_ptr(), b2.data_ptr(), b, t,
                                          c, k, d, 0.1, 0, 0, 1.0, out.data_ptr(), 0, 0.1, 0, 1, st()),
                   "hg_resblock_pair_fwd")
        check_guards(f"pair c{c} k{k} d{d}")
        xf = x.float().transpose(1, 2)
        xa = F.leaky_relu(x.float(), 0.1).bfloat16().float().transpose(1, 2)      # rounded where the kernel rounds
        t1 = F.conv1d(xa, p1.float().permute(1, 2, 0).contiguous(), b1, dilation=d, padding=(k - 1) * d // 2)
        t1 = F.leaky_relu(t1, 0.1).bfloat16().float()
        ref = (F.conv1d(t1, p2.float().permute(1, 2, 0).contiguous(), b2, padding=(k - 1) // 2) + xf).transpose(1, 2)
        assert bool(((out.float() - ref).abs() <= 2.0 ** -8 * ref.abs() + 1.5e-2).all()), (c, k, d)
    print("pair ok", flush=True)


def wgrad():
    from ctypes import c_int
    from hifigan_b200.models import _DiscLayer, _round_up
    for (b, t, cin, cout, k, s, d, pad, g) in ((2, 300, 256, 256, 3, 1, 1, 1, 1), (2, 500, 32, 32, 7, 1, 3, 9, 1),
                                               (2, 400, 64, 64, 3, 1, 1, 1, 1), (2, 300, 128, 256, 41, 2, 1, 20, 16),
                                               (2, 200, 32, 128, 5, 3, 1, 2, 1)):
        gen = torch.Generator().manual_seed(cin + cout + k)
        rows = _round_up(t, s)
        x = torch.zeros(b, rows, cin, dtype=torch.bfloat16, device=dev)
        x[:, :t] = torch.randn(b, t, cin, generator=gen).to(dev).bfloat16()
        t_out = (t + 2 * pad - d * (k - 1) - 1) // s + 1
        dy = torch.randn(b, t_out, cout, generator=gen).to(dev).bfloat16()
        layer = _DiscLayer(cin, cout, k, s, pad, g)
        dwp = guarded((k, cout, layer.cin_tile), torch.float32, torch.zeros(k, cout, layer.cin_tile))
        _lib.check(L.hg_conv1d_wgrad(x.data_ptr(), dy.data_ptr(), b, rows, cin, t_out, t_out, layer.groups_eff, cout, k,
                                     s, d, pad, dwp.data_ptr(), 0, st()), "hg_conv1d_wgrad")
        dw = torch.empty(cout, cin // g, k, dtype=torch.float32, device=dev)
        _lib.check(L.hg_unpack_wgrad_conv(dwp.data_ptr(), cout, cin // g, k, cout, layer.cin_tile, cout // g, layer.merge,
                                          (c_int * k)(*layer.order), dw.data_ptr(), st()))
        check_guards(f"wgrad {cin}->{cout} k{k} s{s}")
        w = torch.zeros(cout, cin // g, k, device=dev, requires_grad=True)
        F.conv1d(x[:, :t].float().transpose(1, 2), w, None, stride=s, padding=pad, dilation=d,
                 groups=g).backward(dy.float().transpose(1, 2))
        assert (dw - w.grad).abs().max().item() <= 2e-3 * w.grad.abs().max().item() + 1e-5
    print("wgrad ok", flush=True)


def mel():
    from oracle import hifigan_oracle as O
    a = O.synthetic_audio(2, 8192 + 77, seed=1)
    for args in ((1024, 80, 22050, 256, 1024, 0, 8000), (512, 40, 16000, 128, 400, 20, None)):
        m = H.mel_spectrogram(a.cuda(), *args).cpu().double()
        ref = O.mel_spectrogram(a.double(), *args)
        assert (m - ref).abs().max().item() < 1e-3
    H.meldataset.flush_range_warnings()
    yc = a.cuda()
    plan = H.meldataset.torch_mels[f"{yc.device}_1024_80_22050_256_1024_0_8000_False"]
    dm = torch.randn(2, 80, plan.frames(yc.shape[1]), device=dev)
    dy = guarded(tuple(yc.shape), torch.float32, torch.zeros(yc.shape))
    mo = guarded((2, 80, plan.frames(yc.shape[1])), torch.float32)
    yg = guarded(tuple(yc.shape), torch.float32, yc)
    _lib.check(L.hg_mel_fwd(plan.handle, yg.data_ptr(), 2, yc.shape[1], mo.data_ptr(), 0, st()), "hg_mel_fwd")
    _lib.check(L.hg_mel_bwd(plan.handle, yg.data_ptr(), dm.data_ptr(), 2, yc.shape[1], dy.data_ptr(), st()), "hg_mel_bwd")
    check_guards("mel fwd / bwd")
    assert (mo.cpu().double() - O.mel_spectrogram(a.double(), 1024, 80, 22050, 256, 1024, 0, 8000)).abs().max().item() < 1e-3
    assert bool(torch.isfinite(dy).all())
    print("mel ok", flush=True)


def ends():
    from oracle import hifigan_oracle as O
    torch.manual_seed(3)
    mpd, msd = H.MultiPeriodDiscriminator().cuda().eval(), H.MultiScaleDiscriminator().cuda().eval()
    y = O.synthetic_audio(1, 2051, seed=2).unsqueeze(1).cuda()
    with torch.no_grad():
        a = mpd(y, y.flip(-1).contiguous())
        b = msd(y, y.flip(-1).contiguous())
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(t).all()) for t in a[0] + a[1] + b[0] + b[1])
    print("ends ok", flush=True)


def step():
    from oracle import hifigan_oracle as O
    from hifigan_b200.train import TrainStep
    h = H.AttrDict(O.config("v1"))
    torch.manual_seed(1234)
    ts = TrainStep(H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator(), h, "cuda")
    ya = O.synthetic_audio(1, 8192, seed=4).cuda()
    out = ts.step(H.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, 8000), ya.unsqueeze(1),
                  H.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, None))
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(v).all()) for v in out.values())
    print("step ok", {k: round(float(v), 4) for k, v in out.items() if k.startswith("loss")}, flush=True)


if __name__ == "__main__":
    fams = sys.argv[1:] or ["conv", "conv2", "pair", "wgrad", "mel", "ends"]
    for f in fams:
        globals()[f]()
    print("sanitize_cases: all requested families ran", flush=True)
