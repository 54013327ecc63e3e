"""Training from a packed int16 corpus on the device: CorpusSampler gives the batches SegmentSampler gives from the
in-memory fp32 pool, bit for bit; the staging kernels write only their outputs and equal their numpy restatement;
the device footprint does not grow with the corpus; train_loop --input_corpus trains, checkpoints and resumes."""
import json

import numpy as np
import pytest
import torch
from scipy.io.wavfile import write

from test_host_corpus import stage_reference

pytestmark = pytest.mark.gpu

SR, SEG = 22050, 8192
MEL = (1024, 80, 256, 1024, SR, 0, 8000)      # n_fft, num_mels, hop, win, sr, fmin, fmax (SegmentSampler's order)
LENGTHS = (30000, 5000, 8192, 12345, 8191, 20000, 9000)     # shorter than, equal to and longer than a segment


@pytest.fixture(scope="module")
def H():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import hifigan_b200
    hifigan_b200._lib.lib()
    return hifigan_b200


def _st():
    return torch.cuda.current_stream().cuda_stream


def _write_wavs(d, lengths, seed):
    rng = np.random.default_rng(seed)
    d.mkdir(exist_ok=True)
    paths = []
    for i, n in enumerate(lengths):
        a = (rng.standard_normal(n) * 4000 * (i + 1) / len(lengths)).clip(-32768, 32767).astype(np.int16)
        if i == 1:
            a[n // 3] = -32768                                   # peak 32768
        p = str(d / f"utt{i}.wav")
        write(p, SR, a)
        paths.append(p)
    return paths


def _write_mels(d, lengths, seed):
    d.mkdir(exist_ok=True)
    g = np.random.default_rng(seed)
    for i, n in enumerate(lengths):
        shape = (1, 80, n // 256 + 1) if i % 2 else (80, n // 256 + 1)
        np.save(d / f"utt{i}.npy", g.standard_normal(shape).astype(np.float32))


@pytest.mark.parametrize("mode", ["peak", "fork", "fine_tuning"])
def test_corpus_sampler_equals_segment_sampler(H, tmp_path, mode):
    """20 consecutive batches, issued without a synchronize (so the two staging slots are reused while earlier
    batches may still be in flight), over the same int16 files, seed and utterance order."""
    from hifigan_b200 import corpus as C
    from hifigan_b200.meldataset import CorpusSampler, SegmentSampler
    from hifigan_b200.train_loop import normalize_fork, normalize_peak, read_wav
    paths = _write_wavs(tmp_path / "wavs", LENGTHS, seed=1)
    ft = mode == "fine_tuning"
    if ft:
        _write_mels(tmp_path / "mels", LENGTHS, seed=2)
    out = str(tmp_path / "train.hgc")
    C.pack(paths, out, SR, mels_dir=str(tmp_path / "mels") if ft else None)
    order = [3, 0, 6, 1, 5, 2, 4]
    prep = {"peak": normalize_peak, "fork": normalize_fork, "fine_tuning": lambda a: a}[mode]
    utts = [prep(read_wav(paths[k], SR) / H.MAX_WAV_VALUE) for k in order]
    mels = [np.load(tmp_path / "mels" / f"utt{k}.npy") for k in order] if ft else None
    n_fft, nm, hop, win, sr, fmin, fmax = MEL
    ref = SegmentSampler(utts, SEG, n_fft, nm, hop, win, sr, fmin, fmax, fmax_loss=None, seed=1234, mels=mels)
    got = CorpusSampler(C.Corpus(out), SEG, n_fft, nm, hop, win, sr, fmin, fmax, fmax_loss=None, seed=1234,
                        normalize=None if ft else mode, fine_tuning=ft, order=order)
    rng = np.random.default_rng(5)
    draws = [rng.integers(0, len(order), int(rng.integers(1, 9))).tolist() for _ in range(20)]
    outs = [got.batch(ix) for ix in draws]                      # no synchronize in between
    refs = [ref.batch(ix) for ix in draws]
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(outs, refs)):
        for name, x, y in zip(("mel", "audio", "mel_loss"), a, b):
            assert x.shape == y.shape and torch.equal(x, y), (i, name)
    assert any(p >= SEG for p in LENGTHS) and any(p < SEG for p in LENGTHS)


def _guarded(shape, dtype, bands, guard=4096):
    n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    raw = torch.full((n + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
    bands.append((raw, guard))
    return raw[guard:guard + n].view(dtype).view(*shape)


@pytest.mark.parametrize("seg", [8192, 8195])         # 16-byte path, and the scalar path for a length not a multiple of 8
def test_stage_kernels_write_only_their_outputs(H, seg):
    """hg_segment_stage_i16 over every int16 value, all three modes and several peaks, and hg_segment_stage_mel with
    partial tiles, each input and output between guard bands of a sentinel byte: the results equal the numpy
    restatement bit for bit (zero past the valid length) and nothing outside a tensor is written."""
    L = H._lib.lib()
    bands = []
    b = 8
    q = np.resize(np.arange(-32768, 32768, dtype=np.int32).astype(np.int16), (b, seg))       # every value at least once
    peaks = np.array([0, 1, 7, 12345, 32767, 32768, 32768, 100], np.int32)
    valid = np.array([seg, seg, seg - 1, 0, 1, seg, 4095, seg], np.int32)
    staged = _guarded((b, seg), torch.int16, bands)
    staged.copy_(torch.from_numpy(q))
    pk = _guarded((b,), torch.int32, bands)
    pk.copy_(torch.from_numpy(peaks))
    vd = _guarded((b,), torch.int32, bands)
    vd.copy_(torch.from_numpy(valid))
    for mode_id, mode in enumerate(("peak", "fork", "none")):
        out = _guarded((b, seg), torch.float32, bands)
        H._lib.check(L.hg_segment_stage_i16(staged.data_ptr(), pk.data_ptr(), vd.data_ptr(), b, seg, mode_id,
                                            out.data_ptr(), _st()), "hg_segment_stage_i16")
        got = out.cpu().numpy()
        for r in range(b):
            want = stage_reference(q[r], int(peaks[r]), mode)
            want[valid[r]:] = 0
            assert np.array_equal(got[r].view(np.int32), want.view(np.int32)), (mode, r)
    for fps, nm in ((32, 80), (33, 100)):
        src = torch.randn(3, fps, nm, generator=torch.Generator().manual_seed(fps))
        vf = np.array([fps, 5, 0], np.int32)
        st = _guarded((3, fps, nm), torch.float32, bands)
        st.copy_(src)
        vfd = _guarded((3,), torch.int32, bands)
        vfd.copy_(torch.from_numpy(vf))
        mo = _guarded((3, nm, fps), torch.float32, bands)
        H._lib.check(L.hg_segment_stage_mel(st.data_ptr(), vfd.data_ptr(), 3, fps, nm, mo.data_ptr(), _st()),
                     "hg_segment_stage_mel")
        want = src.transpose(1, 2).clone()
        for r in range(3):
            want[r, :, vf[r]:] = 0
        assert torch.equal(mo.cpu(), want)
    assert L.hg_segment_stage_i16(staged.data_ptr(), pk.data_ptr(), vd.data_ptr(), b, seg, 3, staged.data_ptr(),
                                  _st()) != 0                                      # unknown mode: refused
    torch.cuda.synchronize()
    for raw, guard in bands:
        assert bool((raw[:guard] == 0xA5).all()) and bool((raw[-guard:] == 0xA5).all()), "write outside a tensor"


def test_device_footprint_does_not_grow_with_the_corpus(H, tmp_path):
    """memory_allocated grows by the same amount for a 20 MB and a 2 GB corpus (batch 16 x 8192, three batches
    held): only the crops reach the device."""
    from hifigan_b200 import corpus as C
    from hifigan_b200.meldataset import CorpusSampler
    n_fft, nm, hop, win, sr, fmin, fmax = MEL
    block = (np.random.default_rng(0).standard_normal(1 << 20) * 3000).astype(np.int16)
    growth = {}
    for label, utt, count in (("20MB", 1 << 20, 10), ("2GB", 1 << 26, 16)):
        path = str(tmp_path / f"{label}.hgc")
        C.write(path, sr, [f"u{i}" for i in range(count)], ((np.tile(block, utt >> 20), None) for _ in range(count)))
        corpus = C.Corpus(path)
        assert corpus.pcm.nbytes == 2 * utt * count
        H.mel_spectrogram(torch.zeros(16, SEG, device="cuda"), n_fft, nm, sr, hop, win, fmin, fmax)   # mel plans
        H.mel_spectrogram(torch.zeros(16, SEG, device="cuda"), n_fft, nm, sr, hop, win, fmin, None)
        H.meldataset.flush_range_warnings()
        torch.cuda.synchronize()
        m0 = torch.cuda.memory_allocated()
        s = CorpusSampler(corpus, SEG, n_fft, nm, hop, win, sr, fmin, fmax, fmax_loss=None, seed=1234)
        held = [s.batch([j % count for j in range(i, i + 16)]) for i in range(3)]
        torch.cuda.synchronize()
        growth[label] = torch.cuda.memory_allocated() - m0
        del held, s, corpus
    assert growth["20MB"] == growth["2GB"], growth
    assert growth["2GB"] < 16 << 20, growth


def _train_args(tmp_path, cp, corpus=None):
    argv = ["--input_wavs_dir", str(tmp_path / "wavs"), "--input_training_file", str(tmp_path / "training.txt"),
            "--input_validation_file", str(tmp_path / "validation.txt"), "--checkpoint_path", str(cp),
            "--config", str(tmp_path / "config_v1.json"), "--stdout_interval", "1", "--checkpoint_interval", "1",
            "--validation_interval", "1000", "--summary_interval", "1000"]
    return argv + (["--input_corpus", str(corpus)] if corpus else [])


def test_train_loop_from_a_packed_corpus(H, tmp_path, monkeypatch):
    """train_loop.main --input_corpus: two steps with g_ / do_ checkpoints, a resume that continues, and a first batch
    bit-identical to the run from the wav files."""
    from hifigan_b200 import corpus as C
    from hifigan_b200 import train_loop
    from hifigan_b200.meldataset import read_filelist
    from hifigan_b200.train import TrainStep
    cfg = dict(H.load_config("v1"))
    cfg.update(batch_size=2, seed=1234, num_gpus=0)
    (tmp_path / "config_v1.json").write_text(json.dumps(cfg))
    lengths = (12000, 7000, 8192, 20000, 9000)
    _write_wavs(tmp_path / "wavs", lengths, seed=9)
    (tmp_path / "training.txt").write_text("\n".join(f"utt{i}|text" for i in range(4)))
    (tmp_path / "validation.txt").write_text("utt4|text")
    corpus = tmp_path / "train.hgc"
    C.pack(read_filelist(str(tmp_path / "training.txt"), str(tmp_path / "wavs")), str(corpus), SR)

    first = {}                                     # run -> (x, y, y_mel) of its first step
    original = TrainStep.step_graphed

    def recording(self, x, y, y_mel, *args, **kwargs):
        first.setdefault(recording.run, (x.clone(), y.clone(), y_mel.clone()))
        return original(self, x, y, y_mel, *args, **kwargs)

    monkeypatch.setattr(TrainStep, "step_graphed", recording)
    recording.run = "wavs"
    train_loop.main(_train_args(tmp_path, tmp_path / "cp_wavs") + ["--training_epochs", "1"])
    recording.run = "corpus"
    cp = tmp_path / "cp"
    r1 = train_loop.main(_train_args(tmp_path, cp, corpus) + ["--training_epochs", "1"])
    assert r1["final_steps"] == 2 and (cp / "g_00000001").exists() and (cp / "do_00000001").exists()
    assert np.isfinite(r1["loss_gen_all"])
    for a, b in zip(first["wavs"], first["corpus"]):
        assert torch.equal(a, b)
    r2 = train_loop.main(_train_args(tmp_path, cp, corpus) + ["--training_epochs", "2"])
    assert r2["final_steps"] == 2 + 2 * 2 and (cp / "g_00000005").exists()     # epoch 0 re-run from step 2, epoch 1
    # a corpus packed from another file list is refused
    (tmp_path / "other.txt").write_text("\n".join(f"utt{i}|text" for i in (1, 0, 2, 3)))
    argv = _train_args(tmp_path, tmp_path / "cp_other", corpus)
    argv[argv.index(str(tmp_path / "training.txt"))] = str(tmp_path / "other.txt")
    with pytest.raises(ValueError, match="was not packed from"):
        train_loop.main(argv + ["--training_epochs", "1"])
