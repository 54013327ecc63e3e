"""The packed int16 corpus on the host (hifigan_b200.corpus): what is packed reads back unchanged, what cannot be
packed is refused, and the staging kernels' three conversions, restated in numpy, equal the host pipeline of the
in-memory path bit for bit."""
import os
import struct
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy.io.wavfile import read, write

from conftest import ROOT
from hifigan_b200 import corpus as C
from hifigan_b200.train_loop import normalize_fork, normalize_peak, read_wav

SR = 22050


def stage_reference(q, m, mode):
    """numpy restatement of hg_segment_stage_i16 for int16 samples q of an utterance with peak m = max|q|."""
    q = np.asarray(q, np.float32)
    if mode == "peak":
        return (q / np.float32(m) * np.float32(0.95)).astype(np.float32) if m > 0 else np.zeros_like(q)
    if mode == "fork":
        return (np.sign(q) * np.float32(0.95)).astype(np.float32)
    return (q * np.float32(2.0 ** -30)).astype(np.float32)


def host_pipeline(path, mode):
    """What train_loop feeds SegmentSampler for one wav file."""
    prep = {"peak": normalize_peak, "fork": normalize_fork, "none": lambda a: a}[mode]
    return prep(read_wav(path, SR) / 32768.0)


def _wavs(tmp_path, specs, seed=0):
    """specs: (name, length, kind) -> int16 wav files under tmp_path/wavs; returns the paths."""
    rng = np.random.default_rng(seed)
    d = tmp_path / "wavs"
    d.mkdir(exist_ok=True)
    paths = []
    for name, n, kind in specs:
        if kind == "zeros":
            a = np.zeros(n, np.int16)
        elif kind == "fullscale":
            a = rng.integers(-32768, 32768, n).astype(np.int16)
            a[n // 2] = -32768
        elif kind == "stereo":
            a = rng.integers(-2000, 2000, (n, 2)).astype(np.int16)
        else:
            a = (rng.standard_normal(n) * 3000).clip(-32768, 32767).astype(np.int16)
        p = str(d / f"{name}.wav")
        write(p, SR, a)
        paths.append(p)
    return paths


SPECS = [("u0", 30000, "noise"), ("u1", 5000, "fullscale"), ("u2", 8192, "zeros"), ("u3", 12345, "stereo"),
         ("u4", 0, "zeros"), ("u5", 1, "noise")]


def test_pack_reads_back_the_wav_files(tmp_path):
    paths = _wavs(tmp_path, SPECS)
    out = str(tmp_path / "train.hgc")
    C.pack(paths, out, SR)
    c = C.Corpus(out)
    assert len(c) == len(SPECS) and c.names == [s[0] for s in SPECS] and c.sampling_rate == SR
    assert c.mels is None and c.num_mels == 0
    for i, p in enumerate(paths):
        sr, ref = read(p)
        ref = ref[:, 0] if ref.ndim > 1 else ref                          # channel 0, as read_wav
        assert sr == SR and c.lengths[i] == ref.size
        assert np.array_equal(c.samples(i), ref)
        assert c.peaks[i] == (int(np.abs(ref.astype(np.int32)).max()) if ref.size else 0)
    assert c.peaks[1] == 32768 and c.peaks[2] == 0
    assert c.offsets[0] == 0 and all(c.offsets[i + 1] == c.offsets[i] + c.lengths[i] for i in range(len(c) - 1))
    assert not c.pcm.flags.writeable
    assert (c.pcm.ctypes.data - c._map.ctypes.data) % C.PAGE == 0


def test_pack_fine_tuning_mels_are_frame_major(tmp_path):
    paths = _wavs(tmp_path, SPECS[:4])
    mels = tmp_path / "mels"
    mels.mkdir()
    g = np.random.default_rng(3)
    ref = {}
    for i, (name, n, _) in enumerate(SPECS[:4]):
        shape = (1, 80, n // 256 + 1) if i % 2 else (80, n // 256 + 1)       # both .npy layouts the reference loads
        ref[name] = g.standard_normal(shape).astype(np.float32)
        np.save(mels / f"{name}.npy", ref[name])
    out = str(tmp_path / "ft.hgc")
    C.pack(paths, out, SR, mels_dir=str(mels))
    c = C.Corpus(out)
    assert c.num_mels == 80 and c.mels.shape == (sum(n // 256 + 1 for _, n, _ in SPECS[:4]), 80)
    for i, (name, n, _) in enumerate(SPECS[:4]):
        assert c.mel_frames[i] == n // 256 + 1
        assert np.array_equal(c.mel(i), ref[name].reshape(80, -1).T)
        assert np.array_equal(c.samples(i), read(paths[i])[1].reshape(n, -1)[:, 0])
    assert (c.mels.ctypes.data - c._map.ctypes.data) % C.PAGE == 0


def test_pack_rejects_other_rates_and_sample_formats(tmp_path):
    d = tmp_path / "w"
    d.mkdir()
    ok = str(d / "ok.wav")
    write(ok, SR, np.zeros(100, np.int16))
    cases = {"rate.wav": (16000, np.zeros(100, np.int16), "16000 SR doesn't match target 22050 SR"),
             "float.wav": (SR, np.zeros(100, np.float32), "not 16-bit PCM"),
             "int32.wav": (SR, np.zeros(100, np.int32), "not 16-bit PCM"),
             "uint8.wav": (SR, np.zeros(100, np.uint8), "not 16-bit PCM")}
    pcm24 = b"\x00\x01\x02" * 100                           # 24-bit PCM (scipy writes no such file)
    (d / "pcm24.wav").write_bytes(b"RIFF" + struct.pack("<I", 36 + len(pcm24)) + b"WAVEfmt " +
                                  struct.pack("<IHHIIHH", 16, 1, 1, SR, SR * 3, 3, 24) + b"data" +
                                  struct.pack("<I", len(pcm24)) + pcm24)
    cases["pcm24.wav"] = (SR, None, "not 16-bit PCM")
    for name, (sr, data, msg) in cases.items():
        p = str(d / name)
        if data is not None:
            write(p, sr, data)
        out = tmp_path / "bad.hgc"
        with pytest.raises(ValueError, match=msg):
            C.pack([ok, p], str(out), SR)
        assert not out.exists() and not os.path.exists(str(out) + ".mels.tmp")    # nothing half-written is left


def test_corpus_refuses_other_files(tmp_path):
    p = tmp_path / "x.hgc"
    p.write_bytes(b"RIFF" + bytes(100))
    with pytest.raises(ValueError, match="not a packed corpus"):
        C.Corpus(str(p))


@pytest.mark.parametrize("m", [0, 1, 7, 12345, 32767, 32768])
def test_stage_modes_restate_the_host_pipeline_exhaustively(m):
    """Every int16 value an utterance of peak m can hold (all 65 536 at m = 32768), through normalize_peak /
    normalize_fork / the fine-tuning path on the values read_wav produces, against the numpy restatement."""
    q = np.arange(-min(m, 32768), min(m, 32767) + 1, dtype=np.int32).astype(np.int16)
    audio = torch.from_numpy(q.astype(np.float32) / np.float32(32768.0)) / 32768.0     # read_wav, then / MAX_WAV_VALUE
    assert int(np.abs(q.astype(np.int32)).max()) == m
    for mode, got in (("peak", normalize_peak(audio)), ("fork", normalize_fork(audio)), ("none", audio)):
        want = stage_reference(q, m, mode)
        assert got.dtype == torch.float32
        assert np.array_equal(got.numpy().view(np.int32), want.view(np.int32)), mode       # bit for bit


def test_stage_reference_equals_host_pipeline_on_packed_files(tmp_path):
    paths = _wavs(tmp_path, SPECS)
    out = str(tmp_path / "train.hgc")
    C.pack(paths, out, SR)
    c = C.Corpus(out)
    for i, p in enumerate(paths):
        if c.lengths[i] == 0:
            continue                                   # normalize_peak cannot take an empty utterance
        for mode in ("peak", "fork", "none"):
            want = host_pipeline(p, mode).numpy()
            got = stage_reference(c.samples(i), int(c.peaks[i]), mode)
            assert np.array_equal(got.view(np.int32), want.view(np.int32)), (p, mode)


def test_pack_command_line_follows_the_file_list(tmp_path):
    import json
    paths = _wavs(tmp_path, SPECS[:3])
    (tmp_path / "training.txt").write_text("u2|c\nu0|a\nu1|b\n")
    (tmp_path / "config.json").write_text(json.dumps({"sampling_rate": SR}))
    out = tmp_path / "train.hgc"
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "hifigan_b200.corpus", "--input_wavs_dir", str(tmp_path / "wavs"),
                        "--input_training_file", str(tmp_path / "training.txt"), "--config",
                        str(tmp_path / "config.json"), "--output", str(out)], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    c = C.Corpus(str(out))
    assert c.names == ["u2", "u0", "u1"]
    assert np.array_equal(c.samples(1), read(paths[0])[1])
