"""The mel front-end at n_fft 256 / 512 / 2048 (the 16 kHz and 44.1 kHz recipes and the other power-of-two STFT
sizes): the forward kernel's lane phases (mel_kernel2<N2>) and the backward kernel's group phases (mel_bwd_kernel<N>),
run on the host through hg_mel_emulate_host / hg_mel_bwd_emulate_host, against the fp64 oracle."""
import ctypes

import numpy as np
import pytest
import torch

from hifigan_b200 import _lib
from oracle import hifigan_oracle as O
from test_oracle_cpu import mel_close

# (n_fft, num_mels, sampling_rate, hop_size, win_size, fmin, fmax)
FWD_CASES = [
    (256, 40, 22050, 64, 256, 50, None),       # hop divides n_fft, fmin > 0
    (256, 80, 16000, 100, 200, 0, 8000),       # hop does not divide n_fft, window shorter than the transform
    (512, 80, 16000, 128, 512, 0, 8000),       # the 16 kHz recipe
    (512, 64, 16000, 160, 400, 30, None),
    (2048, 80, 44100, 512, 2048, 0, None),     # the 44.1 kHz recipe
    (2048, 80, 22050, 300, 1200, 0, 8000),
]
BWD_CASES = [
    (256, 80, 16000, 64, 256, 0, 8000),
    (256, 40, 22050, 100, 200, 50, None),
    (512, 80, 16000, 128, 512, 0, 8000),
    (512, 80, 22050, 160, 400, 0, None),
    (2048, 80, 44100, 512, 2048, 0, None),
    (2048, 80, 22050, 300, 1200, 0, 8000),
]


def _plan(L, case):
    n_fft, nm, sr, hop, win, fmin, fmax = case
    plan = ctypes.c_void_p()
    assert L.hg_mel_plan_create(ctypes.byref(plan), n_fft, nm, sr, hop, win, float(fmin),
                                -1.0 if fmax is None else float(fmax), None) == 0
    return plan


def _audio(t, seed):
    """three items of length t (not a multiple of any hop above); item 1 is silent"""
    y = O.synthetic_audio(3, t, seed=seed)
    y[1] = 0.0
    return y


@pytest.mark.parametrize("case", FWD_CASES, ids=lambda c: "-".join(str(v) for v in c))
def test_mel_sizes_forward_emulation_vs_oracle(case):
    L = _lib.lib()
    plan = _plan(L, case)
    t = 9001
    y = _audio(t, seed=5)
    yn = np.ascontiguousarray(y.numpy())
    frames = L.hg_mel_num_frames(plan, t)
    out = np.zeros((3, case[1], frames), np.float32)
    assert L.hg_mel_emulate_host(plan, yn.ctypes.data, 3, t, out.ctypes.data) == 0
    L.hg_mel_plan_destroy(plan)
    ref = O.mel_spectrogram(y.double(), *case).numpy()
    assert out.shape == ref.shape
    mel_close(out.astype(np.float64), ref, 2e-4)
    assert np.all(out[1] == np.float32(np.log(1e-5)))


@pytest.mark.parametrize("case", BWD_CASES, ids=lambda c: "-".join(str(v) for v in c))
def test_mel_sizes_backward_emulation_vs_autograd(case):
    """forward recompute, complex un-pack, CSR gradient, the Hermitian-packed adjoint transform, window and reflect
    fold-back, against torch autograd through the fp64 oracle mel; the silent item sits below the clamp everywhere and
    gets an exactly zero gradient, and the first and last samples (reflect-padded edges) are compared too"""
    L = _lib.lib()
    t = 7001
    y = _audio(t, seed=4)
    g = torch.Generator().manual_seed(1)
    yd = y.double().requires_grad_(True)
    mel = O.mel_spectrogram(yd, *case)
    dmel = torch.randn(mel.shape, generator=g, dtype=torch.float64)
    (mel * dmel).sum().backward()
    plan = _plan(L, case)
    y32 = np.ascontiguousarray(y.numpy())
    d32 = np.ascontiguousarray(dmel.float().numpy())
    dy = np.zeros_like(y32)
    assert L.hg_mel_bwd_emulate_host(plan, y32.ctypes.data, d32.ctypes.data, 3, t, dy.ctypes.data) == 0
    L.hg_mel_plan_destroy(plan)
    ref = yd.grad.numpy()
    assert np.all(dy[1] == 0.0) and np.all(ref[1] == 0.0)
    pad = (case[0] - case[3]) // 2
    for i in (0, 2):
        scale = np.abs(ref[i]).max()
        err = np.abs(dy[i] - ref[i]).max() / scale
        cos = float(np.dot(dy[i], ref[i]) / (np.linalg.norm(dy[i]) * np.linalg.norm(ref[i])))
        assert err < 2e-3 and cos > 0.99999, (i, err, cos)
        edges = np.r_[0:pad + 1, t - pad - 1:t]
        assert np.abs(dy[i][edges] - ref[i][edges]).max() / scale < 2e-3


def test_mel_backward_rejects_sizes_without_an_fft_path():
    L = _lib.lib()
    for n_fft in (400, 128, 4096):
        plan = _plan(L, (n_fft, 40, 16000, n_fft // 4, n_fft, 0, None))
        y = np.zeros((1, 4 * n_fft), np.float32)
        dmel = np.zeros((1, 40, L.hg_mel_num_frames(plan, y.shape[1])), np.float32)
        dy = np.zeros_like(y)
        assert L.hg_mel_bwd_emulate_host(plan, y.ctypes.data, dmel.ctypes.data, 1, y.shape[1], dy.ctypes.data) != 0
        assert b"256, 512, 1024 or 2048" in L.hg_last_error()
        L.hg_mel_plan_destroy(plan)
