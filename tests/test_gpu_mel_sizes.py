"""The mel front-end at n_fft 256 / 512 / 2048 on the device: mel_kernel2<N2> and mel_bwd_kernel<N> against the fp64
oracle and against their own host emulation, mel_spectrogram under autograd, and whole training steps of the
44.1 kHz (n_fft 2048) and 16 kHz (n_fft 512) recipes against the training oracle."""

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_host_mel_sizes import BWD_CASES, FWD_CASES
from test_oracle_cpu import mel_close

pytestmark = pytest.mark.gpu

LOSS_KEYS = ("loss_disc_f", "loss_disc_s", "loss_mel", "loss_fm_f", "loss_fm_s", "loss_gen_f", "loss_gen_s")


@pytest.fixture(scope="module")
def H():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import hifigan_b200
    hifigan_b200._lib.lib()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return hifigan_b200


def _st():
    return torch.cuda.current_stream().cuda_stream


def _plan(H, y, case):
    H.mel_spectrogram(y, *case)                                             # creates / caches the plan
    n_fft, nm, sr, hop, win, fmin, fmax = case
    return H.meldataset.torch_mels[f"{y.device}_{n_fft}_{nm}_{sr}_{hop}_{win}_{fmin}_{fmax}_False"]


def _audio(t, seed):
    from oracle import hifigan_oracle as O
    y = O.synthetic_audio(3, t, seed=seed)
    y[1] = 0.0
    return y


def _host_forward(H, plan, y):
    L = H._lib.lib()
    yn = np.ascontiguousarray(y.numpy())
    out = np.zeros((y.shape[0], plan.num_mels, plan.frames(y.shape[1])), np.float32)
    H._lib.check(L.hg_mel_emulate_host(plan.handle, yn.ctypes.data, y.shape[0], y.shape[1], out.ctypes.data))
    return out


def _device_backward(H, plan, yc, dmel):
    dy = torch.zeros_like(yc)
    dm = dmel.float().cuda().contiguous()
    H._lib.check(H._lib.lib().hg_mel_bwd(plan.handle, yc.data_ptr(), dm.data_ptr(), yc.shape[0], yc.shape[1],
                                         dy.data_ptr(), _st()), "hg_mel_bwd")
    torch.cuda.synchronize()
    return dy.cpu()


@pytest.mark.parametrize("case", FWD_CASES, ids=lambda c: "-".join(str(v) for v in c))
def test_mel_sizes_forward_vs_oracle_and_emulation(H, case):
    from oracle import hifigan_oracle as O
    t = 9001
    y = _audio(t, seed=5)
    yc = y.cuda()
    got = H.mel_spectrogram(yc, *case).cpu()
    ref = O.mel_spectrogram(y.double(), *case).numpy()
    assert got.shape == ref.shape
    mel_close(got.double().numpy(), ref, 2e-4)
    assert torch.all(got[1] == np.float32(np.log(1e-5)))
    emu = _host_forward(H, _plan(H, yc, case), y)
    mel_close(got.double().numpy(), emu.astype(np.float64), 1e-4)     # same arithmetic; the device contracts to FMAs


@pytest.mark.parametrize("case", BWD_CASES, ids=lambda c: "-".join(str(v) for v in c))
def test_mel_sizes_backward_vs_autograd_and_emulation(H, case):
    from oracle import hifigan_oracle as O
    t = 7001
    y = _audio(t, seed=4)
    yd = y.double().requires_grad_(True)
    mel = O.mel_spectrogram(yd, *case)
    dmel = torch.randn(mel.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    (mel * dmel).sum().backward()
    yc = y.cuda()
    plan = _plan(H, yc, case)
    got, ref = _device_backward(H, plan, yc, dmel), yd.grad
    assert torch.all(got[1] == 0)
    for i in (0, 2):
        assert (got[i] - ref[i]).abs().max() / ref[i].abs().max() < 2e-3
        assert F.cosine_similarity(got[i].double(), ref[i], dim=0).item() > 0.99999
    emu = np.zeros(y.shape, np.float32)
    d32 = np.ascontiguousarray(dmel.float().numpy())
    yn = np.ascontiguousarray(y.numpy())
    H._lib.check(H._lib.lib().hg_mel_bwd_emulate_host(plan.handle, yn.ctypes.data, d32.ctypes.data, 3, t,
                                                      emu.ctypes.data))
    assert np.abs(got.numpy() - emu).max() <= 1e-4 * np.abs(emu).max()     # atomicAdd order differs from the host's


@pytest.mark.parametrize("b,t", [(256, 8192), (8, 262144)])
def test_mel_2048_batch_shapes(H, b, t):
    """cfg5 batch shapes at n_fft 2048: a slice agrees with the oracle, and every item is computed on its own (an item
    run alone gives the same bits as inside the batch)."""
    from oracle import hifigan_oracle as O
    case = (2048, 80, 44100, 512, 2048, 0, None)
    y = O.synthetic_audio(b, t, seed=6).cuda()
    m = H.mel_spectrogram(y, *case)
    frames = (t + 2 * ((2048 - 512) // 2) - 2048) // 512 + 1
    assert m.shape == (b, 80, frames) and bool(torch.isfinite(m).all())
    lo = b - 2
    ref = O.mel_spectrogram(y[lo:].cpu().double(), *case).numpy()
    mel_close(m[lo:].cpu().double().numpy(), ref, 2e-4)
    for i in (0, b // 2, b - 1):
        assert torch.equal(H.mel_spectrogram(y[i:i + 1].contiguous(), *case), m[i:i + 1])
    dmel = torch.randn(m.shape, generator=torch.Generator().manual_seed(2)).cuda()
    plan = _plan(H, y, case)
    dy = torch.zeros_like(y)
    H._lib.check(H._lib.lib().hg_mel_bwd(plan.handle, y.data_ptr(), dmel.data_ptr(), b, t, dy.data_ptr(), _st()))
    dy1 = torch.zeros_like(y[:1])
    H._lib.check(H._lib.lib().hg_mel_bwd(plan.handle, y[b - 1:].data_ptr(), dmel[b - 1:].data_ptr(), 1, t,
                                         dy1.data_ptr(), _st()))
    torch.cuda.synchronize()
    assert bool(torch.isfinite(dy).all())
    assert (dy[b - 1:] - dy1).abs().max().item() <= 1e-5 * dy1.abs().max().item()   # atomicAdd order only


@pytest.mark.parametrize("case", [(256, 40, 16000, 100, 256, 0, 8000), (512, 80, 16000, 128, 400, 0, 8000),
                                  (2048, 80, 44100, 512, 2048, 0, None)])
def test_mel_sizes_write_only_their_outputs(H, case):
    """hg_mel_fwd / hg_mel_bwd with every input and output between two guard bands of a sentinel byte pattern: no
    kernel writes outside its tensor.  The hop does not divide n_fft at 256, and the frame count leaves the last
    block partly empty at every size."""
    from oracle import hifigan_oracle as O
    guard = 4096                                                    # bytes on either side
    bands = []

    def guarded(shape, fill=None):
        n = int(np.prod(shape))
        raw = torch.full((4 * n + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
        t = raw[guard:guard + 4 * n].view(torch.float32).view(*shape)
        if fill is not None:
            t.copy_(fill.reshape(shape))
        bands.append(raw)
        return t

    a = O.synthetic_audio(2, 8192 + 77, seed=1)
    yc = a.cuda()
    plan = _plan(H, yc, case)
    nm, t = case[1], yc.shape[1]
    frames = plan.frames(t)
    yg = guarded((2, t), yc)
    mo = guarded((2, nm, frames))
    dm = guarded((2, nm, frames), torch.randn(2, nm, frames, generator=torch.Generator().manual_seed(5)).cuda())
    dy = guarded((2, t), torch.zeros(2, t, device="cuda"))
    L = H._lib.lib()
    H._lib.check(L.hg_mel_fwd(plan.handle, yg.data_ptr(), 2, t, mo.data_ptr(), 0, _st()), "hg_mel_fwd")
    H._lib.check(L.hg_mel_bwd(plan.handle, yg.data_ptr(), dm.data_ptr(), 2, t, dy.data_ptr(), _st()), "hg_mel_bwd")
    torch.cuda.synchronize()
    for raw in bands:
        assert bool((raw[:guard] == 0xA5).all()) and bool((raw[-guard:] == 0xA5).all()), "write outside a tensor"
    mel_close(mo.cpu().double().numpy(), O.mel_spectrogram(a.double(), *case).numpy(), 2e-4)
    assert bool(torch.isfinite(dy).all())


@pytest.mark.parametrize("n_fft", [256, 512, 2048])
def test_mel_sizes_range_warning_is_lazy_but_kept(H, capsys, n_fft):
    y = torch.zeros(1, 8192, device="cuda")
    y[0, 3000] = -1.5
    H.mel_spectrogram(y, n_fft, 80, 22050, n_fft // 4, n_fft, 0, 8000)
    H.meldataset.flush_range_warnings()
    assert "min value is" in capsys.readouterr().out


@pytest.mark.parametrize("case", [(512, 80, 16000, 128, 512, 0, 8000), (2048, 80, 44100, 512, 2048, 0, None)])
def test_mel_sizes_autograd_vs_oracle(H, case):
    """mel_spectrogram(y) with y.requires_grad (the generated-mel L1 term of the UPSTREAM loop): value and gradient
    against autograd through the fp64 oracle"""
    from oracle import hifigan_oracle as O
    y = O.synthetic_audio(2, 12000, seed=8)
    yd = y.double().requires_grad_(True)
    ref = O.mel_spectrogram(yd, *case)
    w = torch.randn(ref.shape, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    (ref * w).sum().backward()
    yc = y.cuda().requires_grad_(True)
    got = H.mel_spectrogram(yc, *case)
    mel_close(got.detach().cpu().double().numpy(), ref.detach().numpy(), 2e-4)
    (got * w.float().cuda()).sum().backward()
    g, r = yc.grad.cpu().double(), yd.grad
    assert (g - r).abs().max() / r.abs().max() < 2e-3
    assert F.cosine_similarity(g.flatten(), r.flatten(), dim=0).item() > 0.99999


def _recipe(name):
    from oracle import hifigan_oracle as O
    h = dict(O.config("v1"))
    if name == "A":         # 44.1 kHz
        h.update(upsample_rates=[8, 8, 4, 2], upsample_kernel_sizes=[16, 16, 8, 4], n_fft=2048, hop_size=512,
                 win_size=2048, sampling_rate=44100, segment_size=16384, fmax=None)
    else:                   # 16 kHz
        h.update(upsample_rates=[8, 4, 2, 2], upsample_kernel_sizes=[16, 8, 4, 4], n_fft=512, hop_size=128,
                 win_size=512, sampling_rate=16000, segment_size=8192, fmax=8000)
    return h


def _mel_args(h, fmax):
    return (h.n_fft, h.num_mels, h.sampling_rate, h.hop_size, h.win_size, h.fmin, fmax)


@pytest.mark.parametrize("recipe", ["A", "B"])
def test_train_step_recipes_vs_oracle(H, recipe):
    """One TrainStep at batch 2, update=False, against autograd over the training oracle (DESIGN §4 thresholds): the
    seven losses within 2e-2 relative, every parameter gradient cosine >= 0.995 and rel-L2 <= 0.1.  A one-element
    gradient (the weight_g of a discriminator's one-channel conv_post) is one projection of the layer's weight
    gradient that nearly cancels, so bf16 forward noise sets its magnitude at batch 2: those are held to the sign."""
    from oracle import hifigan_oracle as O
    from oracle import train_oracle as TO
    from hifigan_b200.train import TrainStep
    h = H.AttrDict(_recipe(recipe))
    torch.manual_seed(1234)
    nets = (H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator())
    sds = [TO.leaf_params({k: v.detach().clone() for k, v in m.state_dict().items()}) for m in nets]
    ya = O.synthetic_audio(2, h.segment_size, seed=12)
    torch.set_num_threads(max(1, torch.get_num_threads()))
    losses, gg, gp, gs, _, _ = TO.train_step(*sds, h, O.mel_spectrogram(ya, *_mel_args(h, h.fmax)), ya.unsqueeze(1),
                                             O.mel_spectrogram(ya, *_mel_args(h, h.fmax_for_loss)), update=False)
    ts = TrainStep(*nets, h, "cuda")
    yc = ya.cuda()
    out = ts.step(H.mel_spectrogram(yc, *_mel_args(h, h.fmax)), yc.unsqueeze(1),
                  H.mel_spectrogram(yc, *_mel_args(h, h.fmax_for_loss)), update=False)
    for k in LOSS_KEYS:
        assert abs(out[k].item() - losses[k]) <= 2e-2 * abs(losses[k]), (k, out[k].item(), losses[k])
    for net, grads in zip(nets, (gg, gp, gs)):
        for k, p in net.named_parameters():
            got, ref = p.grad.cpu().flatten(), grads[k].flatten()
            cos = F.cosine_similarity(got, ref, dim=0).item()
            rel = ((got - ref).norm() / (ref.norm() + 1e-12)).item()
            assert cos >= 0.995 and (rel <= 0.1 or got.numel() == 1), (k, cos, rel)


def test_graphed_step_matches_eager_recipe_a(H):
    """TrainStep.step_graphed at the 44.1 kHz recipe walks the eager trajectory: losses after 4 steps agree to 1e-3
    relative (fp32 atomics make the two runs non-bit-identical)."""
    from oracle import hifigan_oracle as O
    from hifigan_b200.train import TrainStep
    h = H.AttrDict(_recipe("A"))
    ya = O.synthetic_audio(2, h.segment_size, seed=21).cuda()
    x = H.mel_spectrogram(ya, *_mel_args(h, h.fmax))
    y_mel = H.mel_spectrogram(ya, *_mel_args(h, h.fmax_for_loss))
    res = []
    for graphed in (False, True):
        torch.manual_seed(1234)
        ts = TrainStep(H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator(), h, "cuda")
        for _ in range(4):
            out = (ts.step_graphed if graphed else ts.step)(x, ya.unsqueeze(1), y_mel)
        torch.cuda.synchronize()
        if graphed:
            assert ts.graph_active, "capture fell back to eager"
        res.append({k: out[k].item() for k in LOSS_KEYS})
    for k in LOSS_KEYS:
        assert abs(res[0][k] - res[1][k]) <= 1e-3 * abs(res[0][k]) + 1e-5, (k, res[0][k], res[1][k])


def test_train_driver_recipe_a(H, tmp_path):
    """train_loop.main at the 44.1 kHz recipe on a few synthetic wav files: two steps (the checkpoint after the first),
    g_ / do_ checkpoints, and a finite validation mel error."""
    import json
    from scipy.io.wavfile import write
    from hifigan_b200 import train_loop
    from oracle import hifigan_oracle as O
    cfg = _recipe("A")
    cfg.update(batch_size=2, seed=1234, num_gpus=0)
    (tmp_path / "config.json").write_text(json.dumps(cfg))
    wavs = tmp_path / "wavs"
    wavs.mkdir()
    audio = O.synthetic_audio(3, 30000, seed=9)
    names = [f"utt{i}" for i in range(3)]
    for n, a in zip(names, audio):
        write(wavs / f"{n}.wav", 44100, (a.numpy() * 32767).astype(np.int16))
    (tmp_path / "training.txt").write_text("\n".join(f"{n}|text" for n in names[:2]))
    (tmp_path / "validation.txt").write_text(f"{names[2]}|text")
    cp = tmp_path / "cp"
    r = train_loop.main(["--input_wavs_dir", str(wavs), "--input_training_file", str(tmp_path / "training.txt"),
                         "--input_validation_file", str(tmp_path / "validation.txt"), "--checkpoint_path", str(cp),
                         "--config", str(tmp_path / "config.json"), "--stdout_interval", "1",
                         "--checkpoint_interval", "1", "--validation_interval", "1", "--summary_interval", "1000",
                         "--training_epochs", "2"])
    assert r["final_steps"] == 2 and (cp / "g_00000001").exists() and (cp / "do_00000001").exists()
    assert np.isfinite(r["val_mel_error"]) and np.isfinite(r["loss_gen_all"])
