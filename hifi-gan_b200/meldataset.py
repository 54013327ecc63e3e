"""mel front-end + training-segment sampler — drop-in for the reference's src/meldataset.py.

`mel_spectrogram` keeps the reference signature (meldataset.py:56) and result (log of the HTK power-mel
of a reflect-padded, Hann-windowed STFT, :59-85) but runs as ONE fused sm_100a kernel (hg_mel_fwd) instead
of torchaudio's >= 6 launches.  There is no CPU path: CPU tensors raise.
"""
from __future__ import annotations

import math
import random
from ctypes import byref, c_void_p
from typing import Dict, Optional

import torch

from . import _lib

MAX_WAV_VALUE = 32768.0

# module-level caches, same names as the reference (meldataset.py:50-53)
mel_basis: Dict[str, object] = {}
hann_window: Dict[str, object] = {}
torch_mels: Dict[str, "_MelPlan"] = {}

_pending_range_checks = []


class _MelPlan:
    """Owns one hg_mel_plan (window, twiddles, CSR filterbank) on one device."""

    def __init__(self, device, n_fft, num_mels, sampling_rate, hop_size, win_size, fmin, fmax):
        self.device = device
        self.num_mels = num_mels
        self.handle = c_void_p()
        # ring of (device min/max, pinned host copy) pairs for the lazy range check: allocating pinned memory per
        # call costs more than the kernel for small inputs
        self._ring = [(torch.empty(2, dtype=torch.float32, device=device),
                       torch.empty(2, dtype=torch.float32).pin_memory()) for _ in range(8)]
        self._ring_pos = 0
        self._init = torch.tensor([float("inf"), float("-inf")], dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            _lib.check(_lib.lib().hg_mel_plan_create(byref(self.handle), n_fft, num_mels, sampling_rate,
                                                     hop_size, win_size, float(fmin),
                                                     -1.0 if fmax is None else float(fmax),
                                                     torch.cuda.current_stream().cuda_stream),
                       "hg_mel_plan_create")

    def frames(self, t: int) -> int:
        return _lib.lib().hg_mel_num_frames(self.handle, t)

    def next_minmax(self):
        dev, host = self._ring[self._ring_pos]
        self._ring_pos = (self._ring_pos + 1) % len(self._ring)
        dev.copy_(self._init)
        return dev, host

    def __del__(self):
        try:
            if self.handle:
                _lib.lib().hg_mel_plan_destroy(self.handle)
        except Exception:
            pass


def flush_range_warnings(block: bool = True) -> None:
    """Print the reference's out-of-range messages (meldataset.py:74-77) for finished calls.  The reference
    pays two blocking host syncs per call for this; here the min/max come from a fused reduction and are read
    lazily — on the next call for whatever already finished, or here with block=True."""
    keep = []
    for ev, host in _pending_range_checks:
        if block:
            ev.synchronize()
        elif not ev.query():
            keep.append((ev, host))
            continue
        lo, hi = host[0].item(), host[1].item()
        if lo < -1.:
            print('min value is ', torch.tensor(lo))
        if hi > 1.:
            print('max value is ', torch.tensor(hi))
    _pending_range_checks[:] = keep


def mel_spectrogram(y, n_fft, num_mels, sampling_rate, hop_size, win_size, fmin, fmax, center=False):
    """y [B,T] fp32 on a CUDA device -> [B,num_mels,frames] fp32 (reference meldataset.py:56-85)."""
    if not y.is_cuda:
        raise RuntimeError(f"mel_spectrogram: hifigan_b200 has no CPU path (got {y.device})")
    if center:
        raise NotImplementedError("center=True is never used by the reference (meldataset.py:152-176)")
    mel_key = f'{str(y.device)}_{n_fft}_{num_mels}_{sampling_rate}_{hop_size}_{win_size}_{fmin}_{fmax}_{center}'
    plan = torch_mels.get(mel_key)
    if plan is None:
        plan = _MelPlan(y.device, n_fft, num_mels, sampling_rate, hop_size, win_size, fmin, fmax)
        torch_mels[mel_key] = plan
    squeeze = y.dim() == 1
    y2 = y.reshape(1, -1) if squeeze else y
    if y2.dim() != 2:
        raise ValueError(f"mel_spectrogram expects [B,T], got {tuple(y.shape)}")
    y2 = y2.contiguous()
    if y2.dtype != torch.float32:
        y2 = y2.float()
    b, t = y2.shape
    frames = plan.frames(t)
    if len(_pending_range_checks) >= 6:   # never let a ring slot be reused while its check is pending
        flush_range_warnings(block=True)
    minmax, host = plan.next_minmax()
    stream = torch.cuda.current_stream()
    if torch.is_grad_enabled() and y2.requires_grad:
        # differentiable call (the generated-mel L1 term of the training loss): hg_mel_fwd / hg_mel_bwd as one
        # autograd.Function
        from . import autograd
        out = autograd.mel_forward(y2, plan, minmax.data_ptr())
    else:
        out = torch.empty(b, num_mels, frames, dtype=torch.float32, device=y.device)
        _lib.check(_lib.lib().hg_mel_fwd(plan.handle, y2.data_ptr(), b, t, out.data_ptr(), minmax.data_ptr(),
                                         stream.cuda_stream), "hg_mel_fwd")
    host.copy_(minmax, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(stream)
    _pending_range_checks.append((ev, host))
    flush_range_warnings(block=False)
    return out[0] if squeeze else out


def load_wav(full_path):
    """reference meldataset.py:15-17: (float32 [channels, L] in [-1, 1], sampling_rate), what
    `torchaudio.load(path, normalize=True)` returns.  File IO is outside the accelerated path; when torchaudio has no
    audio backend in the environment the same values are read with scipy (16-/32-bit PCM and float wav files)."""
    try:
        import torchaudio
        data, sampling_rate = torchaudio.load(full_path, normalize=True)
        return data, sampling_rate
    except Exception:  # noqa: BLE001  (no backend / codec: plain PCM reader)
        import numpy as np
        from scipy.io.wavfile import read
        sampling_rate, data = read(full_path)
        data = np.asarray(data)
        if data.dtype == np.int16:
            data = data.astype(np.float32) / 32768.0
        elif data.dtype == np.int32:
            data = data.astype(np.float32) / 2147483648.0
        elif data.dtype == np.uint8:
            data = (data.astype(np.float32) - 128.0) / 128.0
        data = torch.from_numpy(np.ascontiguousarray(data, dtype=np.float32))
        data = data.unsqueeze(0) if data.dim() == 1 else data.t().contiguous()
        return data, sampling_rate


def normalize(audio):
    """Peak normalisation of an utterance — what UPSTREAM's `librosa.util.normalize(audio)` does on a 1-D array.
    (This fork calls it on a [1, L] tensor, where librosa's default axis=0 normalises every SAMPLE by its own magnitude;
    train_loop.normalize_fork reproduces that literal behaviour.  SURVEY.md §8a row S.)"""
    peak = audio.abs().max()
    return audio / peak if peak > 0 else audio


def save_wav(full_path, data, sampling_rate):
    import torchaudio
    torchaudio.save(full_path, data, sampling_rate)


def dynamic_range_compression_torch(x, C=1, clip_val=1e-5):
    return torch.log(torch.clamp(x, min=clip_val) * C)


def dynamic_range_decompression_torch(x, C=1):
    return torch.exp(x) / C


def spectral_normalize_torch(magnitudes):
    return dynamic_range_compression_torch(magnitudes)


def spectral_de_normalize_torch(magnitudes):
    return dynamic_range_decompression_torch(magnitudes)


def read_filelist(list_path, wavs_dir):
    """One `name|text` list file -> wav paths under wavs_dir (reference meldataset.py:88-96)."""
    import os
    with open(list_path, 'r', encoding='utf-8') as fi:
        return [os.path.join(wavs_dir, x.split('|')[0] + '.wav') for x in fi.read().split('\n') if len(x) > 0]


def get_dataset_filelist(a):
    """reference meldataset.py:88-96: `name|text` list files -> wav paths under a.input_wavs_dir."""
    return read_filelist(a.input_training_file, a.input_wavs_dir), read_filelist(a.input_validation_file, a.input_wavs_dir)


class MelDataset(torch.utils.data.Dataset):
    """The reference's `MelDataset` (meldataset.py:99-181): same constructor, same per-item rule and the same
    `(mel, audio, filename, mel_loss)` tuple, with both mel computations on the fused GPU kernel.

    __getitem__ follows the reference line by line — (cached) load, `/ MAX_WAV_VALUE` (the fork's quirk, :128),
    peak normalisation unless fine-tuning (:129-130), sampling-rate check (:132-134), the inclusive
    `random.randint(0, len - seg)` crop or right zero-pad (:141-150), input mel with `fmax` / fine-tuning `.npy` mel
    crop (:152-172), loss mel with `fmax_loss` (:174-176) — using Python's global `random` seeded 1234 at construction
    (:104) so the draw sequence matches the reference's.  Tensors come back on the CPU (what a DataLoader collates);
    the mels are computed on `device` (default: the current CUDA device).  For the training loop's batched,
    GPU-resident form of the same rule see `SegmentSampler`."""

    def __init__(self, training_files, segment_length, n_fft, num_mels, hop_size, win_size, sampling_rate, fmin, fmax,
                 split=True, shuffle=True, n_cache_reuse=1, device=None, fmax_loss=None, fine_tuning=False,
                 base_mels_path=None):
        self.audio_files = training_files
        random.seed(1234)
        if shuffle:
            random.shuffle(self.audio_files)
        self.segment_length = segment_length
        self.sampling_rate = sampling_rate
        self.split = split
        self.n_fft = n_fft
        self.num_mels = num_mels
        self.hop_size = hop_size
        self.win_size = win_size
        self.fmin = fmin
        self.fmax = fmax
        self.fmax_loss = fmax_loss
        self.cached_wav = None
        self.n_cache_reuse = n_cache_reuse
        self._cache_ref_count = 0
        self.device = device
        self.fine_tuning = fine_tuning
        self.base_mels_path = base_mels_path

    def _mel(self, audio, fmax):
        dev = torch.device(self.device) if self.device is not None else torch.device("cuda")
        if dev.type != "cuda":
            raise RuntimeError("MelDataset: hifigan_b200 has no CPU path; pass a CUDA device (or leave device=None)")
        return mel_spectrogram(audio.to(dev), self.n_fft, self.num_mels, self.sampling_rate, self.hop_size,
                               self.win_size, self.fmin, fmax, center=False).cpu()

    def __getitem__(self, index):
        import os
        filename = self.audio_files[index]
        if self._cache_ref_count == 0:
            audio, sampling_rate = load_wav(filename)
            audio = audio / MAX_WAV_VALUE
            if not self.fine_tuning:
                audio = normalize(audio) * 0.95
            self.cached_wav = audio
            if sampling_rate != self.sampling_rate:
                raise ValueError("{} SR doesn't match target {} SR".format(sampling_rate, self.sampling_rate))
            self._cache_ref_count = self.n_cache_reuse
        else:
            audio = self.cached_wav
            self._cache_ref_count -= 1
        audio = torch.as_tensor(audio, dtype=torch.float32).reshape(1, -1)
        if not self.fine_tuning:
            if self.split:
                if audio.size(1) >= self.segment_length:
                    max_audio_start = audio.size(1) - self.segment_length
                    audio_start = random.randint(0, max_audio_start)
                    audio = audio[:, audio_start:audio_start + self.segment_length]
                else:
                    audio = torch.nn.functional.pad(audio, (0, self.segment_length - audio.size(1)), 'constant')
            mel = self._mel(audio, self.fmax)
        else:
            import numpy as np
            mel = torch.from_numpy(np.load(os.path.join(
                self.base_mels_path, os.path.splitext(os.path.split(filename)[-1])[0] + '.npy')))
            if len(mel.shape) < 3:
                mel = mel.unsqueeze(0)
            if self.split:
                frames_per_seg = math.ceil(self.segment_length / self.hop_size)
                if audio.size(1) >= self.segment_length:
                    mel_start = random.randint(0, mel.size(2) - frames_per_seg - 1)
                    mel = mel[:, :, mel_start:mel_start + frames_per_seg]
                    audio = audio[:, mel_start * self.hop_size:(mel_start + frames_per_seg) * self.hop_size]
                else:
                    mel = torch.nn.functional.pad(mel, (0, frames_per_seg - mel.size(2)), 'constant')
                    audio = torch.nn.functional.pad(audio, (0, self.segment_length - audio.size(1)), 'constant')
        mel_loss = self._mel(audio, self.fmax_loss)
        return (mel.squeeze(), audio.squeeze(0), filename, mel_loss.squeeze())

    def __len__(self):
        return len(self.audio_files)


class SegmentSampler:
    """Batched GPU form of MelDataset.__getitem__'s crop/pad rule (reference meldataset.py:141-150):
    utterances live in one resident device pool; a batch is B (utterance, start) pairs drawn with the
    reference's `random.randint(0, len - seg)` rule, gathered into [B, seg] and fed to two fused mel calls
    (input mel with fmax, loss mel with fmax_loss, meldataset.py:152-154,174-176)."""

    def __init__(self, utterances, segment_length, n_fft, num_mels, hop_size, win_size, sampling_rate, fmin,
                 fmax, fmax_loss=None, seed=1234, device="cuda", mels=None):
        """mels: fine-tuning mode (reference meldataset.py:155-172) — one precomputed [num_mels, F_i] (or
        [1, num_mels, F_i]) mel per utterance, e.g. an acoustic model's teacher-forced output loaded from `.npy`; the
        input mel of a batch is then cropped from these instead of being computed from the audio."""
        self.device = torch.device(device)
        self.segment_length = segment_length
        self.hop_size = hop_size
        self.mel_args = (n_fft, num_mels, sampling_rate, hop_size, win_size, fmin)
        self.fmax, self.fmax_loss = fmax, fmax_loss
        self.lengths = [int(u.numel()) for u in utterances]
        self.offsets = [0]
        for n in self.lengths:
            self.offsets.append(self.offsets[-1] + n)
        self.pool = torch.cat([u.reshape(-1).float() for u in utterances]).to(self.device)
        self.rng = random.Random(seed)
        self.fine_tuning = mels is not None
        if self.fine_tuning:
            if len(mels) != len(utterances):
                raise ValueError("SegmentSampler: one mel per utterance is required in fine-tuning mode")
            ms = [torch.as_tensor(m).float().reshape(-1, torch.as_tensor(m).shape[-1]) for m in mels]
            self.mel_frames = [int(m.shape[1]) for m in ms]
            self.mel_offsets = [0]
            for f in self.mel_frames:
                self.mel_offsets.append(self.mel_offsets[-1] + f)
            self.mel_pool = torch.cat(ms, dim=1).to(self.device)          # [num_mels, sum F_i]
            self.frames_per_seg = math.ceil(segment_length / hop_size)

    def draw(self, indices):
        """(pool offset, valid length) per item, following the reference's inclusive randint rule."""
        seg, picks = self.segment_length, []
        for i in indices:
            n = self.lengths[i]
            start = self.rng.randint(0, n - seg) if n >= seg else 0
            picks.append((self.offsets[i] + start, min(n, seg)))
        return picks

    def draw_fine_tuning(self, indices):
        """(audio pool offset, valid samples, mel pool column, valid frames) per item — reference meldataset.py:163-172:
        utterances of at least one segment draw `mel_start = random.randint(0, F - frames_per_seg - 1)` and crop the
        audio at `mel_start * hop`; shorter ones are right-padded with zeros (mel and audio)."""
        seg, fps, hop, picks = self.segment_length, self.frames_per_seg, self.hop_size, []
        for i in indices:
            n, f = self.lengths[i], self.mel_frames[i]
            if n >= seg:
                mel_start = self.rng.randint(0, f - fps - 1)
                a0 = mel_start * hop
                picks.append((self.offsets[i] + a0, max(0, min(n - a0, fps * hop, seg)), self.mel_offsets[i] + mel_start,
                              min(fps, f - mel_start)))
            else:
                picks.append((self.offsets[i], n, self.mel_offsets[i], min(fps, f)))
        return picks

    def _gather(self, indices, picks):
        """The [B, seg] audio crops of drawn `picks` (from draw / draw_fine_tuning for utterances `indices`) and, in
        fine-tuning mode, the [B, num_mels, frames_per_seg] input-mel crops (else None)."""
        seg = self.segment_length
        starts = torch.tensor([p[0] for p in picks], dtype=torch.int64).to(self.device, non_blocking=True)
        valid = torch.tensor([p[1] for p in picks], dtype=torch.int32).to(self.device, non_blocking=True)
        audio = torch.empty(starts.numel(), seg, dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().hg_segment_gather(self.pool.data_ptr(), starts.data_ptr(), valid.data_ptr(), starts.numel(),
                                                seg, audio.data_ptr(), torch.cuda.current_stream().cuda_stream),
                   "hg_segment_gather")
        if not self.fine_tuning:
            return audio, None
        fps = self.frames_per_seg
        col0 = torch.tensor([p[2] for p in picks], dtype=torch.int64, device=self.device)
        nval = torch.tensor([p[3] for p in picks], dtype=torch.int64, device=self.device)
        ar = torch.arange(fps, device=self.device)
        cols = (col0[:, None] + ar[None, :]).clamp_(max=self.mel_pool.shape[1] - 1)      # [B, fps]
        mel = self.mel_pool[:, cols].permute(1, 0, 2) * (ar[None, :] < nval[:, None])[:, None, :]   # zero padding
        return audio, mel.contiguous()

    def batch(self, indices):
        picks = self.draw_fine_tuning(indices) if self.fine_tuning else self.draw(indices)
        audio, mel = self._gather(indices, picks)
        if mel is None:
            mel = mel_spectrogram(audio, *self.mel_args, self.fmax, center=False)
        mel_loss = mel_spectrogram(audio, *self.mel_args, self.fmax_loss, center=False)
        return mel, audio, mel_loss


_STAGE_MODES = {"peak": 0, "fork": 1, None: 2}         # HG_STAGE_PEAK / _FORK / _NONE


class _StagingSlot:
    """A pinned host buffer, its device twin, and the event recorded after the last copy out of the host buffer."""

    def __init__(self, nbytes, device):
        self.host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        self.dev = torch.empty(nbytes, dtype=torch.uint8, device=device)
        self.copied = None


class CorpusSampler(SegmentSampler):
    """`SegmentSampler` over a packed int16 corpus (`hifigan_b200.corpus.Corpus`) that stays on the host: the same
    attributes, the same draw rule (`draw` / `draw_fine_tuning`) and the same two mel calls, but only each batch's
    crops reach the GPU, so the device footprint is O(batch x segment) whatever the corpus size.

    Per batch the host copies the B crops (int16 samples, and in fine-tuning mode the frame-major fp32 mel crops) from
    the memory-mapped corpus into one of two pinned staging slots, one copy moves the slot to the device, and
    hg_segment_stage_i16 / hg_segment_stage_mel turn it into exactly the tensors `SegmentSampler` gathers from its
    in-memory pool over `normalize(read_wav(f) / MAX_WAV_VALUE)`.  An event recorded after each copy guards the slot's
    reuse, so the host prepares batch i + 1 while the device still works on batch i.

    normalize: 'peak' (train_loop.normalize_peak), 'fork' (normalize_fork) or None (fine-tuning, no normalisation).
    order: the corpus entries the sampler's utterance indices 0..n-1 stand for (default: all, in file order)."""

    def __init__(self, corpus, segment_length, n_fft, num_mels, hop_size, win_size, sampling_rate, fmin, fmax,
                 fmax_loss=None, seed=1234, device="cuda", normalize="peak", fine_tuning=False, order=None):
        if normalize not in _STAGE_MODES:
            raise ValueError(f"CorpusSampler: normalize must be 'peak', 'fork' or None, not {normalize!r}")
        if corpus.sampling_rate != sampling_rate:
            raise ValueError("{} SR doesn't match target {} SR".format(corpus.sampling_rate, sampling_rate))
        self.corpus = corpus
        self.device = torch.device(device)
        self.segment_length = segment_length
        self.hop_size = hop_size
        self.num_mels = num_mels
        self.mel_args = (n_fft, num_mels, sampling_rate, hop_size, win_size, fmin)
        self.fmax, self.fmax_loss = fmax, fmax_loss
        self.mode = _STAGE_MODES[normalize]
        order = list(range(len(corpus))) if order is None else list(order)
        self.lengths = corpus.lengths[order].tolist()
        self.offsets = corpus.offsets[order].tolist()          # into corpus.pcm: draw() returns corpus sample offsets
        self.peaks = corpus.peaks[order].tolist()
        self.rng = random.Random(seed)
        self.fine_tuning = fine_tuning
        if fine_tuning:
            if corpus.mels is None:
                raise ValueError(f"CorpusSampler: {corpus.path} holds no fine-tuning mels (pack it with mels_dir)")
            if corpus.num_mels != num_mels:
                raise ValueError(f"CorpusSampler: the corpus mels have {corpus.num_mels} bands, not {num_mels}")
            self.mel_frames = corpus.mel_frames[order].tolist()
            self.mel_offsets = corpus.mel_offsets[order].tolist()
            self.frames_per_seg = math.ceil(segment_length / hop_size)
        self._slots = [None, None]
        self._next = 0

    def _gather(self, indices, picks):
        import numpy as np
        b, seg = len(picks), self.segment_length
        fps = self.frames_per_seg if self.fine_tuning else 0
        audio_bytes = (b * seg * 2 + 255) // 256 * 256
        mel_at = audio_bytes + (3 * b * 4 + 255) // 256 * 256
        total = mel_at + b * fps * self.num_mels * 4
        slot = self._slots[self._next]
        if slot is not None and slot.copied is not None:
            slot.copied.synchronize()                   # the copy that last read this slot has finished
        if slot is None or slot.host.numel() < total:
            slot = self._slots[self._next] = _StagingSlot(total, self.device)
        self._next ^= 1
        host = slot.host.numpy()
        audio_h = host[:b * seg * 2].view(np.int16).reshape(b, seg)
        meta = host[audio_bytes:audio_bytes + 3 * b * 4].view(np.int32).reshape(3, b)     # valid, peak, valid frames
        pcm = self.corpus.pcm
        for j, (i, p) in enumerate(zip(indices, picks)):
            audio_h[j, :p[1]] = pcm[p[0]:p[0] + p[1]]
            meta[0, j], meta[1, j] = p[1], self.peaks[i]
        if self.fine_tuning:
            mel_h = host[mel_at:total].view(np.float32).reshape(b, fps, self.num_mels)
            for j, p in enumerate(picks):
                mel_h[j, :p[3]] = self.corpus.mels[p[2]:p[2] + p[3]]
                meta[2, j] = p[3]
        slot.dev[:total].copy_(slot.host[:total], non_blocking=True)
        slot.copied = torch.cuda.Event()
        slot.copied.record()
        st = torch.cuda.current_stream().cuda_stream
        base = slot.dev.data_ptr()
        audio = torch.empty(b, seg, dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().hg_segment_stage_i16(base, base + audio_bytes + 4 * b, base + audio_bytes, b, seg,
                                                   self.mode, audio.data_ptr(), st), "hg_segment_stage_i16")
        if not self.fine_tuning:
            return audio, None
        mel = torch.empty(b, self.num_mels, fps, dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().hg_segment_stage_mel(base + mel_at, base + audio_bytes + 8 * b, b, fps, self.num_mels,
                                                   mel.data_ptr(), st), "hg_segment_stage_mel")
        return audio, mel
