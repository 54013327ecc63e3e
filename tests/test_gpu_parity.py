"""Parity tests proper: the CUDA path (through the C-ABI / the reference-shaped Python API) against the oracle
and the reference-generated golden fixtures.  Tolerances are stated where they are used.

Declared numerics of the tensor-core path: bf16 operands and bf16-stored activations, fp32 accumulation.
Measured noise floor on random-init weights (profiles/r01_bringup.md): waveform SNR 41-43 dB vs fp32.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from conftest import load_npz  # noqa: E402


@pytest.fixture(scope="module")
def H():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import hifigan_b200
    hifigan_b200._lib.lib()  # the extension must load: there is no fallback
    # torch references in this file must be true fp32 (cuDNN / cuBLAS default to TF32 on this GPU)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return hifigan_b200


@pytest.fixture(scope="module")
def O():
    from oracle import hifigan_oracle
    return hifigan_oracle


def _snr(ref, got):
    return 10 * torch.log10((ref - ref.mean()).pow(2).sum() / (got - ref).pow(2).sum()).item()


# waveform tolerances for the bf16 path
WAVE_MAX_ABS = 2e-3
WAVE_SNR_DB = 35.0


# ----------------------------------------------------------------------------------------------- conv kernel
CONV_CASES = [
    # b, t, cin, cout, k, dil
    (1, 128, 64, 64, 1, 1), (1, 128, 64, 64, 3, 1), (2, 256, 64, 64, 3, 3), (2, 384, 128, 128, 7, 5),
    (1, 512, 256, 256, 11, 5), (3, 200, 128, 256, 3, 1), (2, 256, 32, 32, 3, 1), (2, 256, 32, 32, 11, 5),
    (2, 256, 32, 64, 7, 3), (1, 100, 128, 512, 7, 1), (1, 1, 64, 64, 3, 1), (2, 129, 64, 32, 5, 12),
    (1, 2048, 128, 128, 7, 12),
    # large enough (>= 148 tiles, streamed weights, N >= 128) to take the CTA-pair (cta_group::2) kernel
    (8, 4224, 128, 128, 7, 3), (4, 8192, 256, 256, 3, 1), (2, 10000, 256, 512, 11, 5), (5, 4000, 128, 256, 5, 1),
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv1d_fwd_vs_torch_fp32(H, case):
    """hg_conv1d_fwd on bf16 inputs vs fp32 F.conv1d on the same (bf16-rounded) inputs and weights:
    only accumulation order and the final bf16 rounding differ -> |err| <= 2^-8 * |ref| + eps."""
    from hifigan_b200 import _lib
    L = _lib.lib()
    b, t, cin, cout, k, d = case
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(b, t, cin, generator=g).to(dev).bfloat16()
    w = (torch.randn(cout, cin, k, generator=g) / (cin * k) ** 0.5).to(dev)
    bias = torch.randn(cout, generator=g).to(dev)
    res = [torch.randn(b, t, cout, generator=g).to(dev).bfloat16() for _ in range(3)]
    wp = torch.empty(k, cout, cin, dtype=torch.bfloat16, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(L.hg_pack_conv1d_weight(w.data_ptr(), 0, cout, cin, k, cin, wp.data_ptr(), st))
    out_raw = torch.full((b, t, cout), 7.0, dtype=torch.bfloat16, device=dev)
    out_act = torch.full((b, t, cout), 7.0, dtype=torch.bfloat16, device=dev)
    pad = (k - 1) * d // 2
    _lib.check(L.hg_conv1d_fwd(x.data_ptr(), wp.data_ptr(), bias.data_ptr(), b, t, cin, cout, k, d, pad,
                               res[0].data_ptr(), res[1].data_ptr(), res[2].data_ptr(), 1.0 / 3,
                               out_raw.data_ptr(), out_act.data_ptr(), 0.1, 0, 1, st))
    torch.cuda.synchronize()
    wr = wp.float().permute(1, 2, 0).contiguous()
    ref = F.conv1d(x.float().transpose(1, 2), wr, bias, dilation=d, padding=pad).transpose(1, 2)
    ref = (ref + res[0].float() + res[1].float() + res[2].float()) / 3
    tol = 2.0 ** -8 * ref.abs() + 1e-3
    assert bool(((out_raw.float() - ref).abs() <= tol).all())
    assert bool(((out_act.float() - F.leaky_relu(ref, 0.1)).abs() <= tol).all())


def test_conv1d_rejects_bad_arguments(H):
    from hifigan_b200 import _lib
    L = _lib.lib()
    x = torch.zeros(1, 128, 64, dtype=torch.bfloat16, device="cuda")
    rc = L.hg_conv1d_fwd(x.data_ptr(), x.data_ptr(), 0, 1, 128, 48, 64, 3, 1, 1, 0, 0, 0, 1.0, x.data_ptr(), 0, 0.1, 0, 1, 0)
    assert rc != 0 and b"multiple of 32" in L.hg_last_error()
    rc = L.hg_conv1d_fwd(x.data_ptr(), x.data_ptr(), 0, 1, 128, 64, 64, 41, 5, 1, 0, 0, 0, 1.0, x.data_ptr(), 0, 0.1, 0, 1, 0)
    assert rc != 0 and b"halo" in L.hg_last_error()


PAIR_CASES = [(64, 3, 1), (64, 3, 5), (64, 7, 3), (64, 7, 5), (32, 3, 1), (32, 7, 5), (32, 11, 1), (32, 11, 5)]


@pytest.mark.parametrize("c,k,d", PAIR_CASES)
@pytest.mark.parametrize("b,t", [(2, 500), (1, 118), (3, 1)])
def test_resblock_pair_vs_torch_fp32(H, c, k, d, b, t):
    """hg_resblock_pair_fwd (fused conv-lrelu-conv-residual) vs fp32 torch on the same bf16-rounded inputs,
    with the intermediate rounded to bf16 exactly where the kernel rounds it.  Covers ragged T (not a multiple
    of the 129-k row tile), T smaller than one tile and T == 1."""
    from hifigan_b200 import _lib
    L = _lib.lib()
    assert L.hg_resblock_pair_supported(c, k, d) == 1
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(c * 1000 + k * 10 + d)
    x = torch.randn(b, t, c, generator=g).to(dev).bfloat16()
    w1 = (torch.randn(c, c, k, generator=g) / (c * k) ** 0.5).to(dev)
    w2 = (torch.randn(c, c, k, generator=g) / (c * k) ** 0.5).to(dev)
    b1, b2 = torch.randn(c, generator=g).to(dev), torch.randn(c, generator=g).to(dev)
    r1 = torch.randn(b, t, c, generator=g).to(dev).bfloat16()
    r2 = torch.randn(b, t, c, generator=g).to(dev).bfloat16()
    st = torch.cuda.current_stream().cuda_stream
    wp1 = torch.empty(k, c, c, dtype=torch.bfloat16, device=dev)
    wp2 = torch.empty(k, c, c, dtype=torch.bfloat16, device=dev)
    _lib.check(L.hg_pack_conv1d_weight(w1.data_ptr(), 0, c, c, k, c, wp1.data_ptr(), st))
    _lib.check(L.hg_pack_conv1d_weight(w2.data_ptr(), 0, c, c, k, c, wp2.data_ptr(), st))
    out_raw = torch.full((b, t, c), 7.0, dtype=torch.bfloat16, device=dev)
    out_act = torch.full((b, t, c), 7.0, dtype=torch.bfloat16, device=dev)
    _lib.check(L.hg_resblock_pair_fwd(x.data_ptr(), wp1.data_ptr(), b1.data_ptr(), wp2.data_ptr(), b2.data_ptr(),
                                      b, t, c, k, d, 0.1, r1.data_ptr(), r2.data_ptr(), 1.0 / 3,
                                      out_raw.data_ptr(), out_act.data_ptr(), 0.01, 0, 1, st))
    torch.cuda.synchronize()
    xa = F.leaky_relu(x.float(), 0.1).bfloat16().float().transpose(1, 2)
    t1 = F.conv1d(xa, wp1.float().permute(1, 2, 0).contiguous(), b1, dilation=d, padding=(k - 1) * d // 2)
    t1 = F.leaky_relu(t1, 0.1).bfloat16().float()
    y = F.conv1d(t1, wp2.float().permute(1, 2, 0).contiguous(), b2, padding=(k - 1) // 2).transpose(1, 2)
    ref = (y + x.float() + r1.float() + r2.float()) / 3
    # one bf16 ulp of the output + the effect of 1-ulp flips of the bf16 intermediate
    tol = 2.0 ** -8 * ref.abs() + 1.5e-2
    assert bool(((out_raw.float() - ref).abs() <= tol).all())
    assert bool(((out_act.float() - F.leaky_relu(ref, 0.01)).abs() <= tol).all())
    assert (out_raw.float() - ref).abs().mean().item() < 2e-3


@pytest.mark.parametrize("c,k,d", [(64, 3, 1), (64, 7, 12), (64, 5, 6), (32, 3, 2), (32, 7, 12), (32, 5, 2)])
@pytest.mark.parametrize("b,t", [(2, 700), (1, 130), (3, 1)])
def test_resblock_single_vs_torch_fp32(H, c, k, d, b, t):
    """hg_resblock_pair_fwd with w2 == NULL: one ResBlock2 step (lrelu -> dilated conv -> + x) vs fp32 torch."""
    from hifigan_b200 import _lib
    L = _lib.lib()
    assert L.hg_resblock_single_supported(c, k, d) == 1
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(c * 1000 + k * 10 + d)
    x = torch.randn(b, t, c, generator=g).to(dev).bfloat16()
    w1 = (torch.randn(c, c, k, generator=g) / (c * k) ** 0.5).to(dev)
    b1 = torch.randn(c, generator=g).to(dev)
    r1 = torch.randn(b, t, c, generator=g).to(dev).bfloat16()
    st = torch.cuda.current_stream().cuda_stream
    wp1 = torch.empty(k, c, c, dtype=torch.bfloat16, device=dev)
    _lib.check(L.hg_pack_conv1d_weight(w1.data_ptr(), 0, c, c, k, c, wp1.data_ptr(), st))
    out_raw = torch.full((b, t, c), 7.0, dtype=torch.bfloat16, device=dev)
    out_act = torch.full((b, t, c), 7.0, dtype=torch.bfloat16, device=dev)
    _lib.check(L.hg_resblock_pair_fwd(x.data_ptr(), wp1.data_ptr(), b1.data_ptr(), 0, 0, b, t, c, k, d, 0.1,
                                      r1.data_ptr(), 0, 0.5, out_raw.data_ptr(), out_act.data_ptr(), 0.1, 0, 1, st))
    torch.cuda.synchronize()
    xa = F.leaky_relu(x.float(), 0.1).bfloat16().float().transpose(1, 2)
    y = F.conv1d(xa, wp1.float().permute(1, 2, 0).contiguous(), b1, dilation=d, padding=(k - 1) * d // 2)
    ref = (y.transpose(1, 2) + x.float() + r1.float()) * 0.5
    tol = 2.0 ** -8 * ref.abs() + 2e-3
    assert bool(((out_raw.float() - ref).abs() <= tol).all())
    assert bool(((out_act.float() - F.leaky_relu(ref, 0.1)).abs() <= tol).all())


@pytest.mark.parametrize("ver", ["v1", "v3"])
def test_fused_and_unfused_generator_paths_agree(H, O, ver):
    """The Generator through fused ResBlock pairs vs the same Generator through two-launch convs."""
    from hifigan_b200 import models
    h = H.AttrDict(O.config(ver))
    torch.manual_seed(1234)
    G = H.Generator(h).cuda().eval()
    x = torch.randn(2, 80, 40, device="cuda")
    with torch.no_grad():
        a = G(x).clone()
        models._FUSE_PAIRS = False
        try:
            b = G(x).clone()
        finally:
            models._FUSE_PAIRS = True
    assert (a - b).abs().max().item() < 1e-3 and _snr(b.cpu(), a.cpu()) > 38.0


@pytest.mark.parametrize("k,u", [(16, 8), (4, 2), (8, 4)])
def test_polyphase_conv_transpose_vs_torch(H, k, u):
    from hifigan_b200.models import _PackedConv, _conv
    from hifigan_b200 import _lib
    dev = torch.device("cuda")
    cin, cout, b, t = 128, 64, 2, 200
    torch.manual_seed(k)
    m = torch.nn.ConvTranspose1d(cin, cout, k, u, padding=(k - u) // 2).to(dev)
    pc = _PackedConv(m, "convtr", dev)
    pc.refresh()
    x = torch.randn(b, t, cin, device=dev).bfloat16()
    out = torch.empty(b, t * u, cout, dtype=torch.bfloat16, device=dev)
    _conv(_lib.lib(), x, pc, b, t, out_raw=out)
    torch.cuda.synchronize()
    wr = m.weight.detach().bfloat16().float()
    ref = F.conv_transpose1d(x.float().transpose(1, 2), wr, m.bias, stride=u, padding=(k - u) // 2).transpose(1, 2)
    assert bool(((out.float() - ref).abs() <= 2.0 ** -8 * ref.abs() + 1e-3).all())


# ------------------------------------------------------------------------------------------------- generator
@pytest.mark.parametrize("ver", ["tiny", "tiny2"])
def test_generator_small_vs_reference_golden(H, ver):
    """Full state_dict + input + the REFERENCE's own output from tests/golden (generated by make_golden.py)."""
    from oracle import hifigan_oracle as O
    z = load_npz(f"gen_{ver}.npz")
    G = H.Generator(H.AttrDict(O.config(ver)))
    G.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")})
    G = G.cuda().eval()
    with torch.no_grad():
        y = G(torch.from_numpy(z["x"]).cuda()).cpu()
    ref = torch.from_numpy(z["y"])
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() < WAVE_MAX_ABS and _snr(ref, y) > WAVE_SNR_DB


@pytest.mark.parametrize("ver", ["v1", "v2", "v3"])
def test_generator_full_size_vs_reference_golden(H, O, ver):
    """Same-seed construction (bit-identical weights, tests/test_host_cpu.py) + the reference's stored output,
    with weight_norm attached, after remove_weight_norm(), and with weight_g x3 (tanh in its non-linear range)."""
    z = load_npz(f"gen_{ver}_seed1234.npz")
    torch.manual_seed(1234)
    G = H.Generator(H.AttrDict(O.config(ver))).cuda().eval()
    x = torch.from_numpy(z["x"]).cuda()
    ref = torch.from_numpy(z["y"])
    # V2's 8..64-channel layers average far fewer bf16 rounding errors per output than V1/V3: its measured
    # bf16 noise floor on random-init weights is ~32 dB (V1: 42.5 dB, profiles/r01_bringup.md)
    snr_min = 28.0 if ver == "v2" else WAVE_SNR_DB
    with torch.no_grad():
        y = G(x).cpu().clone()
        assert (y - ref).abs().max().item() < WAVE_MAX_ABS and _snr(ref, y) > snr_min
        sd3 = {k: (v * 3 if k.endswith("weight_g") else v) for k, v in G.state_dict().items()}
        G.load_state_dict(sd3)
        y3 = G(x).cpu().clone()
        ref3 = torch.from_numpy(z["y_g3"])
        # saturated regime: errors are amplified by the x3^N gain before tanh squashes them; compare loosely
        assert (y3 - ref3).abs().mean().item() < 0.05
        G.load_state_dict({k: (v / 3 if k.endswith("weight_g") else v) for k, v in G.state_dict().items()})
        G.remove_weight_norm()
        y2 = G(x).cpu()
        assert (y2 - ref).abs().max().item() < WAVE_MAX_ABS and _snr(ref, y2) > snr_min


def test_generator_batch_and_ragged_lengths(H, O):
    """Batch items are independent and any frame count works (F not a multiple of the 128-row tile)."""
    h = H.AttrDict(O.config("v3"))
    torch.manual_seed(1234)
    G = H.Generator(h).cuda().eval()
    sd = {k: v.detach().cpu() for k, v in G.state_dict().items()}
    torch.manual_seed(3)
    for b, frames in [(1, 1), (3, 7), (2, 45)]:
        x = torch.randn(b, 80, frames)
        with torch.no_grad():
            y = G(x.cuda()).cpu()
            ref = O.generator_forward(sd, h, x)
        assert y.shape == ref.shape == (b, 1, frames * 256)
        assert (y - ref).abs().max().item() < WAVE_MAX_ABS
    # linearity in the batch dimension: permuting items permutes outputs exactly
    x = torch.randn(4, 80, 16).cuda()
    with torch.no_grad():
        a = G(x).clone()
        bperm = G(x.flip(0)).flip(0)
    assert torch.equal(a, bperm)


def test_generator_full_config2_properties(H, O):
    """BASELINE config 2 size (64 x 80x1024): too big for the CPU oracle, so check size-independent properties:
    every batch item equals the same item computed alone, and time-tiles are consistent with a shorter run
    on the overlap (fully convolutional, receptive field +-13 frames: SURVEY §5)."""
    h = H.AttrDict(O.config("v1"))
    torch.manual_seed(1234)
    G = H.Generator(h).cuda().eval()
    G.remove_weight_norm()
    torch.manual_seed(0)
    x = torch.randn(64, 80, 1024, device="cuda")
    with torch.no_grad():
        y = G(x).clone()
        assert y.shape == (64, 1, 262144) and bool(torch.isfinite(y).all())
        y5 = G(x[5:6].contiguous()).clone()
        assert torch.equal(y[5:6], y5)
        ys = G(x[9:10, :, 256:512].contiguous()).clone()  # frames 256..511 alone
    lo, hi = (256 + 16) * 256, (512 - 16) * 256
    inner = y[9, 0, lo:hi]
    assert (inner - ys[0, 0, 16 * 256:-16 * 256]).abs().max().item() < 1e-6
    assert 0.003 < y.std().item() < 0.1


def test_standalone_resblocks_vs_oracle(H, O):
    torch.manual_seed(7)
    for cls, key, dil in ((H.ResBlock1, "1", (1, 3, 5)), (H.ResBlock2, "2", (2, 6))):
        blk = cls(None, 64, 7, dil)
        sd = {"resblocks.0." + k: v.detach() for k, v in blk.state_dict().items()}
        x = torch.randn(2, 64, 300)
        fwd = O.resblock1_forward if key == "1" else O.resblock2_forward
        with torch.no_grad():
            ref = fwd(sd, "resblocks.0", x, 7, dil)
            y = blk.cuda()(x.cuda()).cpu()
        assert (y - ref).abs().max().item() < 0.05 and _snr(ref, y) > 38.0


# ------------------------------------------------------------------------------------------------------- mel
@pytest.mark.parametrize("name", ["y", "special", "odd"])
@pytest.mark.parametrize("fmax", [8000, None])
def test_mel_vs_reference_golden(H, name, fmax):
    from test_oracle_cpu import mel_close
    z = load_npz("mel.npz")
    got = H.mel_spectrogram(torch.from_numpy(z[name]).cuda(), 1024, 80, 22050, 256, 1024, 0, fmax).cpu().numpy()
    ref = z[f"mel_{name}_fmax{fmax}"]
    assert got.shape == ref.shape
    mel_close(got.astype(np.float64), ref, 2e-4)  # fp32 kernel vs fp32 torchaudio: log-domain 2e-4


def test_mel_matches_its_host_emulation_bitwise_enough(H):
    """GPU kernel vs the same phase functions run on the host: differences only from FMA contraction."""
    import ctypes
    from hifigan_b200 import _lib
    from oracle import hifigan_oracle as O
    y = O.synthetic_audio(3, 20000, seed=11)
    L = _lib.lib()
    plan = ctypes.c_void_p()
    assert L.hg_mel_plan_create(ctypes.byref(plan), 1024, 80, 22050, 256, 1024, 0.0, 8000.0, None) == 0
    yn = np.ascontiguousarray(y.numpy())
    frames = L.hg_mel_num_frames(plan, 20000)
    out = np.zeros((3, 80, frames), np.float32)
    assert L.hg_mel_emulate_host(plan, yn.ctypes.data, 3, 20000, out.ctypes.data) == 0
    got = H.mel_spectrogram(y.cuda(), 1024, 80, 22050, 256, 1024, 0, 8000).cpu().numpy()
    assert np.abs(got - out).max() < 1e-4


def test_mel_large_batch_properties(H, O):
    """cfg5 sizes (B=256 x 8192 and 8 x 262144): item independence + agreement with the oracle on a slice."""
    y = O.synthetic_audio(256, 8192, seed=5).cuda()
    m = H.mel_spectrogram(y, 1024, 80, 22050, 256, 1024, 0, 8000)
    assert m.shape == (256, 80, 32)
    m7 = H.mel_spectrogram(y[7:8].contiguous(), 1024, 80, 22050, 256, 1024, 0, 8000)
    assert torch.equal(m[7:8], m7)
    ref = O.mel_spectrogram(y[250:].cpu().double(), 1024, 80, 22050, 256, 1024, 0, 8000)
    assert (m[250:].cpu().double() - ref).abs().max().item() < 1e-3
    long = O.synthetic_audio(8, 262144, seed=6).cuda()
    ml = H.mel_spectrogram(long, 1024, 80, 22050, 256, 1024, 0, None)
    assert ml.shape == (8, 80, 1024) and bool(torch.isfinite(ml).all())


def test_mel_range_warning_is_lazy_but_kept(H, capsys):
    y = torch.zeros(1, 8192, device="cuda")
    y[0, 100] = 1.5
    H.mel_spectrogram(y, 1024, 80, 22050, 256, 1024, 0, 8000)
    H.meldataset.flush_range_warnings()
    assert "max value is" in capsys.readouterr().out


@pytest.mark.parametrize("hop,win,t,b", [(100, 1024, 9001, 3), (250, 1000, 22050, 2), (255, 1024, 8192, 5),
                                         (512, 512, 70001, 1), (1024, 1024, 40000, 2), (256, 1024, 8190, 4),
                                         (64, 1024, 5000, 2)])
def test_mel_unaligned_hops_and_lengths(H, O, hop, win, t, b):
    """The fused n_fft = 1024 kernel stages its input with 16-byte cp.async copies when (length, hop) allow and
    4-byte ones otherwise, and a block's last frames may be missing: hop sizes / lengths on both sides of every one
    of those conditions against the fp64 oracle (log domain, bins within 60 dB of the frame peak, 2e-4)."""
    y = O.synthetic_audio(b, t, seed=hop + t)
    ref = O.mel_spectrogram(y.double(), 1024, 80, 22050, hop, win, 0, 8000)
    got = H.mel_spectrogram(y.cuda(), 1024, 80, 22050, hop, win, 0, 8000).cpu().double()
    assert got.shape == ref.shape
    loud = ref > ref.max(dim=1, keepdim=True).values - 13.8
    assert (got - ref).abs()[loud].max().item() < 2e-4


@pytest.mark.parametrize("case", range(4))
def test_mel_other_shapes_vs_reference_golden(H, case):
    """mel_spectrogram at the shapes of the reference's other callers (SURVEY §8f-4: n_fft != 1024, 16 kHz, fmax None,
    win < n_fft, fmin > 0) — the direct-DFT kernel against outputs of the reference's own function."""
    from test_oracle_cpu import mel_close
    z = load_npz("mel_other.npz")
    n_fft, nm, sr, hop, win, fmin, fmax = [int(v) for v in z["cases"][case]]
    y = torch.from_numpy(z["y"]).cuda()
    got = H.mel_spectrogram(y, n_fft, nm, sr, hop, win, fmin, None if fmax < 0 else fmax)
    ref = z[f"mel_{case}"]
    assert tuple(got.shape) == ref.shape
    mel_close(got.cpu().double().numpy(), ref, 2e-4)


def test_segment_sampler_batch(H, O):
    from hifigan_b200.meldataset import SegmentSampler
    utts = [O.synthetic_audio(1, n, seed=n)[0] for n in (30000, 5000, 8192, 12345)]
    s = SegmentSampler(utts, 8192, 1024, 80, 256, 1024, 22050, 0, 8000, fmax_loss=None, seed=1234)
    import random
    ref_rng = random.Random(1234)
    mel, audio, mel_loss = s.batch([0, 1, 2, 3])
    assert audio.shape == (4, 8192) and mel.shape == (4, 80, 32) and mel_loss.shape == (4, 80, 32)
    for i, u in enumerate(utts):
        start = ref_rng.randint(0, u.numel() - 8192) if u.numel() >= 8192 else 0
        want = O.crop_or_pad_segment(u.unsqueeze(0), 8192, start)[0]
        assert torch.equal(audio[i].cpu(), want)
    ref = O.mel_spectrogram(audio.cpu().double(), 1024, 80, 22050, 256, 1024, 0, None)
    assert (mel_loss.cpu().double() - ref).abs().max().item() < 1e-3


def test_segment_sampler_fine_tuning_batch(H, O):
    """fine-tuning mode (meldataset.py:155-172): input mels cropped from precomputed per-utterance mels at the drawn
    frame, audio cropped at frame * hop, short utterances zero-padded — bit-exact against the oracle's restatement."""
    import random
    from hifigan_b200.meldataset import SegmentSampler
    lens = (30000, 5000, 8192, 12345)
    utts = [O.synthetic_audio(1, n, seed=n)[0] for n in lens]
    g = torch.Generator().manual_seed(3)
    mels = [torch.randn(1, 80, n // 256 + 1, generator=g) for n in lens]
    s = SegmentSampler(utts, 8192, 1024, 80, 256, 1024, 22050, 0, 8000, fmax_loss=None, seed=99,
                       mels=[m.numpy() for m in mels])
    ref_rng = random.Random(99)
    mel, audio, mel_loss = s.batch([0, 1, 2, 3])
    assert audio.shape == (4, 8192) and mel.shape == (4, 80, 32) and mel_loss.shape == (4, 80, 32)
    for i, (u, m) in enumerate(zip(utts, mels)):
        start = ref_rng.randint(0, m.shape[2] - 32 - 1) if u.numel() >= 8192 else 0
        wm, wa = O.finetune_crop_or_pad(m, u.unsqueeze(0), 8192, 256, start)
        wa = torch.nn.functional.pad(wa, (0, 8192 - wa.shape[1]))       # a crop that runs past the end (see draw rule)
        assert torch.equal(audio[i].cpu(), wa[0]) and torch.equal(mel[i].cpu(), wm[0])
    ref = O.mel_spectrogram(audio.cpu().double(), 1024, 80, 22050, 256, 1024, 0, None)
    assert (mel_loss.cpu().double() - ref).abs().max().item() < 1e-3


# --------------------------------------------------------------------------------------------- discriminators
GENERAL_CASES = [
    # b, t_in, cin, cout, k, stride, pad, groups
    (3, 300, 32, 128, 5, 3, 2, 1),      # DiscriminatorP layer 1 shape class (KC=32, residue boxes)
    (2, 911, 128, 512, 5, 3, 2, 1),
    (2, 100, 512, 1024, 5, 3, 2, 1),
    (2, 51, 1024, 1024, 5, 1, 2, 1),
    (2, 1000, 128, 128, 41, 2, 20, 4),   # DiscriminatorS grouped / strided layers
    (2, 600, 128, 256, 41, 2, 20, 16),   # 8-channel groups -> merged block-diagonal tiles
    (1, 700, 256, 512, 41, 4, 20, 16),
    (1, 515, 512, 1024, 41, 4, 20, 16),
    (1, 130, 1024, 1024, 41, 1, 20, 16),
]


@pytest.mark.parametrize("case", GENERAL_CASES)
def test_general_conv_vs_torch(H, case):
    """hg_conv1d_general_fwd (strided through residue boxes, grouped through per-group N tiles) vs fp32
    F.conv1d on the same bf16-rounded inputs and weights."""
    from hifigan_b200 import _lib
    from hifigan_b200.models import _DiscLayer, _round_up
    L = _lib.lib()
    b, t, cin, cout, k, s, pad, g = case
    dev = torch.device("cuda")
    gen = torch.Generator().manual_seed(sum(case))
    rows = _round_up(t, s)
    x = torch.zeros(b, rows, cin, dtype=torch.bfloat16, device=dev)
    x[:, :t] = torch.randn(b, t, cin, generator=gen).to(dev).bfloat16()
    w = (torch.randn(cout, cin // g, k, generator=gen) / (cin // g * k) ** 0.5).to(dev).bfloat16().float()
    bias = torch.randn(cout, generator=gen).to(dev)
    layer = _DiscLayer(cin, cout, k, s, pad, g)
    wp = layer.pack(w)
    t_out = (t + 2 * pad - k) // s + 1
    rows_out = t_out + 5
    out = torch.full((b, rows_out, cout), 7.0, dtype=torch.bfloat16, device=dev)
    _lib.check(L.hg_conv1d_general_fwd(x.data_ptr(), wp.data_ptr(), bias.data_ptr(), b, rows, cin, t_out, rows_out,
                                       layer.groups_eff, cout, k, s, pad, out.data_ptr(), 0.1, 0, 0, 0,
                                       torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = F.leaky_relu(F.conv1d(x[:, :t].float().transpose(1, 2), w, bias, stride=s, padding=pad, groups=g), 0.1)
    ref = ref.transpose(1, 2)
    assert ref.shape[1] == t_out
    assert bool(((out[:, :t_out].float() - ref).abs() <= 2.0 ** -8 * ref.abs() + 2e-3).all())
    assert bool((out[:, t_out:] == 7.0).all())  # pitch rows are left untouched


def test_disc_end_kernels_vs_torch(H):
    from hifigan_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda")
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(9)
    for (b, t, period, k, s, pad, cout) in [(3, 8192, 1, 15, 1, 7, 128), (2, 8192, 3, 5, 3, 2, 32),
                                             (2, 1000, 7, 5, 3, 2, 32), (2, 4097, 1, 15, 1, 7, 128)]:
        y = torch.randn(b, t, generator=g).to(dev)
        w = torch.randn(cout, k, generator=g).to(dev) * 0.3
        bias = torch.randn(cout, generator=g).to(dev)
        tp = (t + period - 1) // period * period
        hin = tp // period
        hout = (hin + 2 * pad - k) // s + 1
        out = torch.zeros(b * period, hout + 2, cout, dtype=torch.bfloat16, device=dev)
        _lib.check(L.hg_disc_first_conv_fwd(y.data_ptr(), w.data_ptr(), bias.data_ptr(), b, t, period, k, s, pad, cout,
                                            hout + 2, out.data_ptr(), 0.1, st))
        yp = F.pad(y.unsqueeze(1), (0, tp - t), "reflect") if tp != t else y.unsqueeze(1)
        x4 = yp.view(b, 1, hin, period)
        ref = F.leaky_relu(F.conv2d(x4, w.view(cout, 1, k, 1), bias, stride=(s, 1), padding=(pad, 0)), 0.1)
        got = out[:, :hout].float().view(b, period, hout, cout).permute(0, 3, 2, 1)
        assert (got - ref).abs().max().item() < 2.0 ** -7 * ref.abs().max().item() + 1e-3
    # last conv
    x = torch.randn(6, 55, 1024, generator=g).to(dev).bfloat16()
    w = torch.randn(1024, 3, generator=g).to(dev) * 0.05
    bias = torch.randn(1, generator=g).to(dev)
    out = torch.empty(6, 51, dtype=torch.float32, device=dev)
    _lib.check(L.hg_disc_last_conv_fwd(x.data_ptr(), w.data_ptr(), bias.data_ptr(), 6, 51, 55, 1024, 3, out.data_ptr(), st))
    ref = F.conv1d(x[:, :51].float().transpose(1, 2), w.unsqueeze(0), bias, padding=1)[:, 0]
    assert (out - ref).abs().max().item() < 2e-3
    # avg pool incl. odd length and the 0.5-weighted edges
    for t in (8192, 4097, 9):
        y = torch.randn(2, t, generator=g).to(dev)
        out = torch.empty(2, t // 2 + 1, device=dev)
        _lib.check(L.hg_avgpool_4_2_2_fwd(y.data_ptr(), 2, t, out.data_ptr(), st))
        assert torch.allclose(out, F.avg_pool1d(y.unsqueeze(1), 4, 2, padding=2)[:, 0], atol=1e-6)


def _seeded_discs(H, O):
    torch.manual_seed(1234)
    H.Generator(H.AttrDict(O.config("v1")))
    return H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator()


def test_discriminators_vs_reference_golden(H, O):
    """MPD / MSD forward on the CUDA path vs the REFERENCE's stored logits, feature-map magnitudes and losses
    (tests/golden/disc_seed1234.npz; MSD in train mode so the spectral-norm power iterations are exercised).
    bf16 operands: logits within 3e-2 abs, losses within 2 % rel."""
    z = load_npz("disc_seed1234.npz")
    mpd, msd = _seeded_discs(H, O)
    mpd, msd = mpd.cuda().eval(), msd.cuda().train()
    y, y_hat = torch.from_numpy(z["y"]).cuda(), torch.from_numpy(z["y_hat"]).cuda()
    with torch.no_grad():
        for name, D in (("mpd", mpd), ("msd", msd)):
            rs, gs, fr, fg = D(y, y_hat)
            for i, (r, g) in enumerate(zip(rs, gs)):
                ref_r, ref_g = z[f"{name}_logits_r{i}"], z[f"{name}_logits_g{i}"]
                assert tuple(r.shape) == ref_r.shape
                assert np.abs(r.cpu().numpy() - ref_r).max() < 3e-2 * max(1.0, np.abs(ref_r).max())
                assert np.abs(g.cpu().numpy() - ref_g).max() < 3e-2 * max(1.0, np.abs(ref_g).max())
            mags = np.array([[float(f.abs().mean()) for f in fl] + [0.0] * (8 - len(fl)) for fl in fr])
            assert np.allclose(mags, z[f"{name}_fmap_abs_mean_r"], rtol=2e-2, atol=1e-4)
            fl = H.feature_loss(fr, fg).item()
            assert abs(fl - float(z[f"{name}_feature_loss"])) < 2e-2 * abs(float(z[f"{name}_feature_loss"]))
            dl, rl, gl = H.discriminator_loss(rs, gs)
            assert abs(dl.item() - float(z[f"{name}_disc_loss"])) < 2e-2 * abs(float(z[f"{name}_disc_loss"]))
            gt, _ = H.generator_loss(gs)
            assert abs(gt.item() - float(z[f"{name}_gen_loss"])) < 2e-2 * abs(float(z[f"{name}_gen_loss"]))


def test_discriminator_fmaps_vs_oracle(H, O):
    """Every one of the 54 feature maps against the fp32 oracle on the same weights (odd length: reflect pad)."""
    mpd, msd = _seeded_discs(H, O)
    sd_p = {k: v.detach().clone() for k, v in mpd.state_dict().items()}
    sd_s = {k: v.detach().clone() for k, v in msd.state_dict().items()}
    y = O.synthetic_audio(2, 8000, seed=21).unsqueeze(1)
    y_hat = O.synthetic_audio(2, 8000, seed=22).unsqueeze(1)
    torch.set_num_threads(8)
    with torch.no_grad():
        ref_p = O.mpd_forward(sd_p, y, y_hat)
        ref_s = O.msd_forward(sd_s, y, y_hat, train=False)
        got_p = mpd.cuda().eval()(y.cuda(), y_hat.cuda())
        got_s = msd.cuda().eval()(y.cuda(), y_hat.cuda())
    for ref, got in ((ref_p, got_p), (ref_s, got_s)):
        for fl_ref, fl_got in zip(ref[2] + ref[3], got[2] + got[3]):
            assert len(fl_ref) == len(fl_got)
            for fr, fg in zip(fl_ref, fl_got):
                assert fr.shape == fg.shape
                scale = fr.abs().max().item() + 1e-6
                assert (fg.cpu() - fr).abs().max().item() < 4e-2 * scale


def test_training_step_forward_losses_vs_reference_golden(H, O):
    """Forward half of the UPSTREAM training step (G, mel of the generated audio, both D passes, all seven loss
    terms) vs the REFERENCE's values (tests/golden/train_fwd_seed1234.npz).  Tolerance: 3 % relative on every
    loss (bf16 operands; the adversarial terms are sums over 8 sub-discriminators of O(1) values)."""
    from hifigan_b200.train import step_losses
    z = load_npz("train_fwd_seed1234.npz")
    h = H.AttrDict(O.config("v1"))
    torch.manual_seed(1234)
    G = H.Generator(h).cuda().train()
    mpd = H.MultiPeriodDiscriminator().cuda().train()
    msd = H.MultiScaleDiscriminator().cuda().train()
    audio = torch.from_numpy(z["audio"]).cuda()
    x = H.mel_spectrogram(audio, 1024, 80, 22050, 256, 1024, 0, 8000)
    y_mel = H.mel_spectrogram(audio, 1024, 80, 22050, 256, 1024, 0, None)
    out = step_losses(G, mpd, msd, x, audio.unsqueeze(1), y_mel, h)
    ref_wave = torch.from_numpy(z["y_g_hat"])
    assert (out["y_g_hat"].cpu() - ref_wave).abs().max().item() < WAVE_MAX_ABS
    for k in ("loss_disc_f", "loss_disc_s", "loss_mel", "loss_fm_f", "loss_fm_s", "loss_gen_f", "loss_gen_s"):
        ref = float(z[k])
        assert abs(out[k].item() - ref) < 3e-2 * abs(ref), (k, out[k].item(), ref)


def test_loss_sum_kernel(H):
    from hifigan_b200 import _lib
    g = torch.Generator().manual_seed(4)
    a, b = torch.randn(3, 1000, 37, generator=g).cuda(), torch.randn(3, 1000, 37, generator=g).cuda()
    assert torch.allclose(H.feature_loss([[a]], [[b]]), 2 * (a - b).abs().mean(), rtol=1e-5)
    l, r, gg = H.discriminator_loss([a], [b])
    assert torch.allclose(l, ((1 - a) ** 2).mean() + (b ** 2).mean(), rtol=1e-5) and isinstance(r[0], float)
    assert torch.allclose(H.generator_loss([a])[0], ((1 - a) ** 2).mean(), rtol=1e-5)


def test_inference_e2e_driver_matches_per_file_reference_schedule(H, O, tmp_path):
    """hifigan_b200.inference (SURVEY §8f-1): the batched, length-bucketed mel -> wav driver writes the same int16
    samples as the reference's per-file schedule (src/inference_e2e.py:45-56: generator(x) -> * 32768 -> astype
    int16), with the reference's output names; checkpoint + config.json layout as src/inference.py:74-80."""
    import json
    from scipy.io.wavfile import read
    from hifigan_b200 import inference as drv
    cfg = dict(O.config("v3"))
    cfg["seed"] = 1234
    h = H.AttrDict(cfg)
    torch.manual_seed(3)
    G = H.Generator(h)
    cp = tmp_path / "cp"
    cp.mkdir()
    torch.save({"generator": G.state_dict()}, cp / "g_00000001")
    (cp / "config.json").write_text(json.dumps(cfg))
    mels = tmp_path / "mels"
    mels.mkdir()
    g = torch.Generator().manual_seed(0)
    frames = {"u0": 40, "u1": 33, "u2": 40, "u3": 40, "u4": 33}
    data = {k: torch.randn(1, 80, f, generator=g) for k, f in frames.items()}
    for k, v in data.items():
        np.save(mels / f"{k}.npy", v.numpy())
    out = tmp_path / "out"
    drv.main(["e2e", "--checkpoint_file", str(cp / "g_00000001"), "--input_mels_dir", str(mels), "--output_dir", str(out),
              "--max_batch", "2"])
    Gd = G.cuda().eval()
    Gd.remove_weight_norm()
    for k, v in data.items():
        sr, wav = read(out / f"{k}_generated_e2e.wav")
        with torch.no_grad():
            ref = (Gd(v.cuda()).squeeze() * 32768.0).cpu().numpy().astype("int16")
        assert sr == h.sampling_rate and wav.dtype == np.int16 and wav.shape == ref.shape
        assert np.array_equal(wav, ref), k


def _int16_close(wav, ref_float, what):
    """written int16 samples vs the ORACLE's fp32 waveform under the declared bf16 numerics: max |diff| <= 5e-3 of
    full scale (SURVEY §8d waveform tolerance) and SNR >= 35 dB against the reference's own `* 32768 -> int16`"""
    ref = (ref_float * 32768.0).astype("int16")
    assert wav.dtype == np.int16 and wav.shape == ref.shape, what
    diff = wav.astype(np.float64) - ref.astype(np.float64)
    assert np.abs(diff).max() <= 5e-3 * 32768, (what, np.abs(diff).max())
    sig = ref.astype(np.float64) - ref.astype(np.float64).mean()
    snr = 10 * np.log10((sig ** 2).sum() / max((diff ** 2).sum(), 1e-9))
    assert snr >= 35.0, (what, snr)


def test_inference_drivers_vs_oracle(H, O, tmp_path):
    """Both inference drivers against the ORACLE (not this repo's own Generator): `e2e` mode on .npy mels of three
    different lengths (src/inference_e2e.py:34-57) and `wav` mode on wav files (src/inference.py:37-62), including the
    reference's quirk of dividing torchaudio's already-normalised floats by 32768 again (inference.py:51-52) — the
    mel the Generator sees is that of the 32768-times-quieter signal."""
    import json
    from scipy.io.wavfile import read, write
    from hifigan_b200 import inference as drv
    cfg = dict(O.config("v1"))
    cfg["seed"] = 1234
    h = H.AttrDict(cfg)
    torch.manual_seed(11)
    G = H.Generator(h)
    sd = {k: v.detach().clone() for k, v in G.state_dict().items()}
    cp = tmp_path / "cp"
    cp.mkdir()
    torch.save({"generator": G.state_dict()}, cp / "g_00000001")
    (cp / "config.json").write_text(json.dumps(cfg))
    # ---- mel -> wav
    mels = tmp_path / "mels"
    mels.mkdir()
    audio = {"a": O.synthetic_audio(1, 9000, seed=1), "b": O.synthetic_audio(1, 5000, seed=2),
             "c": O.synthetic_audio(1, 9000, seed=3)}
    data = {k: O.mel_spectrogram(v, 1024, 80, 22050, 256, 1024, 0, 8000) for k, v in audio.items()}
    for k, v in data.items():
        np.save(mels / f"{k}.npy", v.numpy())
    out = tmp_path / "out_e2e"
    drv.main(["e2e", "--checkpoint_file", str(cp / "g_00000001"), "--input_mels_dir", str(mels), "--output_dir", str(out)])
    for k, v in data.items():
        sr, wav = read(out / f"{k}_generated_e2e.wav")
        with torch.no_grad():
            ref = O.generator_forward(sd, h, v).squeeze().numpy()
        assert sr == h.sampling_rate
        _int16_close(wav, ref, k)
    # ---- wav -> mel -> wav
    wavs = tmp_path / "wavs"
    wavs.mkdir()
    for k, v in audio.items():
        write(wavs / f"{k}.wav", 22050, (v[0].numpy() * 32767).astype(np.int16))
    out = tmp_path / "out_wav"
    drv.main(["wav", "--checkpoint_file", str(cp / "g_00000001"), "--input_wavs_dir", str(wavs), "--output_dir", str(out)])
    for k, v in audio.items():
        sr, wav = read(out / f"{k}_generated.wav")
        pcm = torch.from_numpy((v[0].numpy() * 32767).astype(np.int16).astype(np.float32) / 32768.0)   # load_wav
        x = O.mel_spectrogram((pcm / 32768.0).unsqueeze(0), 1024, 80, 22050, 256, 1024, 0, 8000)       # the quirk
        with torch.no_grad():
            ref = O.generator_forward(sd, h, x).squeeze().numpy()
        _int16_close(wav, ref, k + " (wav mode)")


def test_meldataset_class_matches_reference_rule(H, O, tmp_path):
    """`MelDataset` (reference meldataset.py:99-181): constructor signature, the `(mel, audio, filename, mel_loss)`
    tuple, the seeded shuffle and inclusive randint crop / right zero-pad, both mels against the oracle."""
    import random
    from scipy.io.wavfile import write
    files = []
    lengths = [20000, 6000, 8192, 12345]
    for i, n in enumerate(lengths):
        a = O.synthetic_audio(1, n, seed=40 + i)[0]
        path = str(tmp_path / f"f{i}.wav")
        write(path, 22050, (a.numpy() * 32767).astype(np.int16))
        files.append(path)
    ds = H.MelDataset(list(files), 8192, 1024, 80, 256, 1024, 22050, 0, 8000, n_cache_reuse=0, shuffle=True,
                      fmax_loss=None, device="cuda")
    # the reference's bookkeeping, replayed: seed, shuffle, then one randint per long-enough item
    random.seed(1234)
    expect = list(files)
    random.shuffle(expect)
    assert ds.audio_files == expect and len(ds) == 4
    state = random.getstate()
    items = [ds[i] for i in range(4)]
    random.setstate(state)
    from scipy.io.wavfile import read
    for (mel, audio, name, mel_loss), path in zip(items, expect):
        _, pcm = read(path)
        a = torch.from_numpy(pcm.astype(np.float32) / 32768.0) / 32768.0            # load_wav, then the / MAX_WAV_VALUE quirk
        a = a / a.abs().max() * 0.95                                                  # normalize(audio) * 0.95
        if a.numel() >= 8192:
            s0 = random.randint(0, a.numel() - 8192)
            seg = a[s0:s0 + 8192]
        else:
            seg = torch.nn.functional.pad(a, (0, 8192 - a.numel()))
        assert name == path and audio.shape == (8192,) and mel.shape == (80, 32) and mel_loss.shape == (80, 32)
        assert torch.allclose(audio, seg, atol=1e-7)
        for got, fmax in ((mel, 8000), (mel_loss, None)):
            ref = O.mel_spectrogram(seg.double().unsqueeze(0), 1024, 80, 22050, 256, 1024, 0, fmax)[0]
            lin_g, lin_r = got.double().exp(), ref.exp()       # fp32 kernel: relative in the power domain, with a
            assert bool(((lin_g - lin_r).abs() <= 2e-3 * lin_r + 1e-6 * lin_r.max()).all())   # floor 60 dB below the peak
    with pytest.raises(ValueError, match="SR doesn't match"):
        H.MelDataset([files[0]], 8192, 1024, 80, 256, 1024, 16000, 0, 8000, shuffle=False)[0]


@pytest.mark.parametrize("ver", ["v1", "v3"])
def test_ragged_batch_is_bit_identical_to_per_item_calls(H, O, ver):
    """`Generator(x, lengths=...)`: utterances of different lengths stacked in one call give, for every item, exactly
    the samples of that item run alone (the reference's schedule, src/inference.py:55) — every layer treats the rows
    past an item's end as zero padding.  Lengths straddle the 128-row tiles of every stage; the padded tails hold
    garbage mel values on purpose."""
    h = H.AttrDict(O.config(ver))
    torch.manual_seed(21)
    G = H.Generator(h).cuda().eval()
    G.remove_weight_norm()
    frames = [37, 5, 64, 23, 1, 50]
    g = torch.Generator().manual_seed(2)
    x = torch.randn(len(frames), 80, max(frames), generator=g).cuda()
    hop = 256
    with torch.no_grad():
        y = G(x, lengths=torch.tensor(frames))
        for i, f in enumerate(frames):
            alone = G(x[i:i + 1, :, :f].contiguous())
            assert torch.equal(y[i, 0, : f * hop], alone[0, 0]), (ver, i, f)
        # and a second ragged call with other lengths through the same workspaces (stale tails must not leak)
        frames2 = [64, 64, 2, 9, 33, 17]
        y2 = G(x, lengths=torch.tensor(frames2))
        for i, f in enumerate(frames2):
            alone = G(x[i:i + 1, :, :f].contiguous())
            assert torch.equal(y2[i, 0, : f * hop], alone[0, 0]), (ver, "second", i, f)
    with torch.no_grad(), pytest.raises(ValueError):
        G(x, lengths=torch.tensor([1, 2, 3]))


def test_randomised_shapes_sweep():
    """tests/gpu_fuzz.py, fixed seed: batch sizes, frame counts, audio lengths, (n_fft, hop, win) and training batch
    sizes the fixed cases above do not hit — generators, discriminators (logits + all feature maps), mel and one
    full training step (losses + every gradient) against the oracle, with the fixed tests' tolerances."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tests", "gpu_fuzz.py"), "0", "8"], capture_output=True,
                         text=True, cwd=root, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "failures: 0" in out.stdout


def test_bench_dump_outputs_is_what_the_generator_returns(H, tmp_path):
    """`bench.py --dump-outputs DIR` after `--steps 2` of the cfg1 workload (V1, 1 x 80 x 256 mel from seed 0, weights
    from seed 1234, weight_norm folded) writes the waveform a caller of Generator gets for the same input."""
    import json
    import subprocess
    import sys
    from hifigan_b200.configs import load_config
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dump = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--workload", "cfg1", "--steps", "2", "--warmup", "1",
           "--no-cpu-baseline", "--dump-outputs", str(dump)]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=root, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    assert sorted(os.listdir(dump)) == ["y_g_hat.npy"]
    got = np.load(dump / "y_g_hat.npy")
    torch.manual_seed(1234)
    G = H.Generator(load_config("v1")).cuda().eval()
    G.remove_weight_norm()
    torch.manual_seed(0)
    x = torch.randn(1, 80, 256)
    with torch.no_grad():
        ref = G(x.cuda()).cpu().numpy()
    assert got.dtype == np.float32 and got.shape == ref.shape == (1, 1, 65536)
    assert np.abs(got - ref).max() <= 1e-6
