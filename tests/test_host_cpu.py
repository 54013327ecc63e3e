"""Host-side logic that needs no GPU: the module/state_dict contract, same-seed construction against the
reference-generated fingerprints, the C-ABI surface, the mel kernel's arithmetic through its host emulation."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import hifigan_b200 as H
from conftest import ROOT, load_npz
from hifigan_b200 import _lib
from oracle import hifigan_oracle as O


def _stats(sd):
    keys = sorted(sd)
    return np.array([[float(sd[k].double().sum()), float(sd[k].double().abs().sum()), sd[k].numel()] for k in keys]), keys


@pytest.mark.parametrize("ver", ["v1", "v2", "v3"])
def test_same_seed_construction_matches_reference(ver):
    """torch.manual_seed(1234); Generator(h) must reproduce the reference's parameters bit for bit: the RNG draw
    order (incl. init_weights' no-op normal_ draws, SURVEY App. B.4) is part of the contract."""
    z = load_npz(f"gen_{ver}_seed1234.npz")
    torch.manual_seed(1234)
    G = H.Generator(H.AttrDict(O.config(ver)))
    stats, keys = _stats(G.state_dict())
    assert keys == list(z["sd_keys"])
    assert np.array_equal(stats, z["sd_stats"])


def test_discriminator_same_seed_construction():
    z = load_npz("disc_seed1234.npz")
    torch.manual_seed(1234)
    H.Generator(H.AttrDict(O.config("v1")))
    mpd, msd = H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator()
    for name, D in (("mpd", mpd), ("msd", msd)):
        stats, keys = _stats(D.state_dict())
        assert keys == list(z[f"{name}_sd_keys"])
        assert np.array_equal(stats, z[f"{name}_sd_stats"])


def test_state_dict_contract_v1():
    G = H.Generator(H.AttrDict(O.config("v1")))
    sd = G.state_dict()
    assert len(sd) == 234  # SURVEY §8a row G
    assert tuple(sd["conv_pre.weight_g"].shape) == (512, 1, 1) and tuple(sd["conv_pre.weight_v"].shape) == (512, 80, 7)
    assert tuple(sd["ups.0.weight_g"].shape) == (512, 1, 1)  # ConvTranspose: dim 0 = input channel
    assert tuple(sd["ups.0.weight_v"].shape) == (512, 256, 16)
    assert "resblocks.11.convs2.2.weight_v" in sd and tuple(sd["conv_post.weight_v"].shape) == (1, 32, 7)
    assert sum(p.numel() for p in G.parameters()) == 13936130
    G.remove_weight_norm()
    sd2 = G.state_dict()
    assert "conv_pre.weight" in sd2 and not any(k.endswith("weight_g") for k in sd2)
    assert sum(p.numel() for p in G.parameters()) == 13926017


def test_state_dict_contract_v3_and_discriminators():
    G = H.Generator(H.AttrDict(O.config("v3")))
    assert "resblocks.0.convs.1.weight_g" in G.state_dict()
    assert sum(p.numel() for p in G.parameters()) == 1464322
    mpd, msd = H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator()
    assert len(mpd.state_dict()) == 90 and len(msd.state_dict()) == 80
    assert sum(p.numel() for p in mpd.parameters()) == 41105770
    assert "discriminators.0.convs.1.weight_orig" in msd.state_dict()
    assert "discriminators.0.convs.1.weight_u" in dict(msd.named_buffers())
    assert tuple(mpd.state_dict()["discriminators.4.convs.3.weight_v"].shape) == (1024, 512, 5, 1)


def test_resblock_selector_is_a_string_compare():
    h = H.AttrDict(O.config("tiny"))
    h.resblock = 1  # int, not '1'  -> ResBlock2, exactly like the reference (models.py:82)
    G = H.Generator(h)
    assert type(G.resblocks[0]).__name__ == "ResBlock2"


def test_load_reference_style_checkpoint(tmp_path):
    z = load_npz("gen_tiny.npz")
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")}
    path = tmp_path / "g_00000001"
    H.save_checkpoint(str(path), {"generator": sd})
    G = H.Generator(H.AttrDict(O.config("tiny")))
    G.load_state_dict(H.load_checkpoint(str(path), "cpu")["generator"])
    for k, v in G.state_dict().items():
        assert torch.equal(v, sd[k])
    assert H.scan_checkpoint(str(tmp_path), "g_") == str(path)
    assert H.scan_checkpoint(str(tmp_path), "do_") is None
    with pytest.raises(AssertionError):
        H.load_checkpoint(str(tmp_path / "missing"), "cpu")


def test_no_cpu_path():
    G = H.Generator(H.AttrDict(O.config("tiny"))).eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        G(torch.zeros(1, 80, 8))
    with pytest.raises(RuntimeError, match="no CPU path"):
        H.mel_spectrogram(torch.zeros(1, 8192), 1024, 80, 22050, 256, 1024, 0, 8000)
    with pytest.raises(RuntimeError, match="no CPU path"):
        H.MultiScaleDiscriminator()(torch.zeros(1, 1, 64), torch.zeros(1, 1, 64))
    with pytest.raises(RuntimeError, match="no CPU path"):
        H.MultiPeriodDiscriminator()(torch.zeros(1, 1, 64), torch.zeros(1, 1, 64))


def test_helpers():
    assert H.get_padding(11, 5) == 25 and H.get_padding(3) == 1
    h = H.AttrDict({"a": 1})
    h.b = 2
    assert h["b"] == 2 and h.a == 1
    assert H.LRELU_SLOPE == 0.1 and H.MAX_WAV_VALUE == 32768.0


def test_losses_have_no_cpu_path():
    """The three loss functions run on hg_loss_sum / hg_loss_grad only: CPU tensors raise instead of silently falling
    back to torch ops (their values are checked against the oracle on the GPU, tests/test_gpu_parity.py)."""
    g = torch.Generator().manual_seed(0)
    fr = [[torch.randn(2, 4, 9, generator=g)]]
    dr = [torch.randn(2, 7, generator=g)]
    with pytest.raises(RuntimeError, match="no CPU path"):
        H.feature_loss(fr, fr)
    with pytest.raises(RuntimeError, match="no CPU path"):
        H.discriminator_loss(dr, dr)
    with pytest.raises(RuntimeError, match="no CPU path"):
        H.generator_loss(dr)


# ------------------------------------------------------------------------------------------- C-ABI surface
def test_library_exports_every_declared_symbol_at_abi_4():
    header = open(os.path.join(ROOT, "include", "hifigan_b200.h")).read()
    declared = set(re.findall(r"\b(hg_[a-z0-9_]+)\s*\(", header))
    declared -= {"hg_mel_plan"}
    lib = ctypes.CDLL(_lib.build())
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/hifigan_b200.h but not exported"
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    # ABI 3 dropped the first three entry points (ABI 2 had them), ABI 4 the last two
    for name in ("hg_set_cta_limit", "hg_unpack_wgrad_convtr", "hg_l1_sum_bf16", "hg_fold_weight_norm",
                 "hg_wgrad_finish_convtr"):
        assert not hasattr(lib, name), f"{name} is still exported"
    assert _lib.lib().hg_abi_version() == 4


def test_unpack_wgrad_rejects_a_row_larger_than_shared_memory():
    """hg_unpack_wgrad_conv stages one [cin_g][k] row in shared memory (at most 96 KB): a larger row is refused
    before anything reaches the device."""
    from ctypes import c_int
    L = _lib.lib()
    order = (c_int * 41)(*range(41))
    fake = 256                      # never dereferenced: the check comes first
    assert L.hg_unpack_wgrad_conv(fake, 8, 600, 41, 8, 600, 8, 1, order, fake, None) != 0
    assert b"hg_unpack_wgrad_conv: row of 24600 values does not fit" in L.hg_last_error()


def test_convtr_geometry():
    from ctypes import byref, c_int
    L = _lib.lib()
    for k, u, pad, want in [(16, 8, 4, (3, -1)), (4, 2, 1, (3, -1)), (8, 4, 2, (3, -1)), (3, 1, 1, (3, -1)),
                            (4, 4, 0, (1, 0))]:
        n, s = c_int(), c_int()
        assert L.hg_convtr1d_geometry(k, u, pad, byref(n), byref(s)) == 0
        assert (n.value, s.value) == want
    assert L.hg_convtr1d_geometry(0, 1, 0, None, None) != 0
    assert b"bad arguments" in L.hg_last_error()


@pytest.mark.parametrize("name", ["y", "special", "odd"])
@pytest.mark.parametrize("fmax", [8000, None])
def test_mel_kernel_arithmetic_on_host_vs_reference(name, fmax):
    """hg_mel_emulate_host runs the CUDA kernel's own phase functions (Stockham radix-8 FFT, real un-packing,
    CSR mel, log-clamp) with threads serialised; it must reproduce the reference-generated fixtures."""
    from test_oracle_cpu import mel_close
    z = load_npz("mel.npz")
    L = _lib.lib()
    plan = ctypes.c_void_p()
    assert L.hg_mel_plan_create(ctypes.byref(plan), 1024, 80, 22050, 256, 1024, 0.0,
                                -1.0 if fmax is None else float(fmax), None) == 0
    y = np.ascontiguousarray(z[name])
    b, t = y.shape
    frames = L.hg_mel_num_frames(plan, t)
    out = np.zeros((b, 80, frames), np.float32)
    assert L.hg_mel_emulate_host(plan, y.ctypes.data, b, t, out.ctypes.data) == 0
    L.hg_mel_plan_destroy(plan)
    ref = z[f"mel_{name}_fmax{fmax}"]
    assert out.shape == ref.shape
    mel_close(out.astype(np.float64), ref, 2e-4)


def test_mel_plan_rejects_unsupported():
    L = _lib.lib()
    plan = ctypes.c_void_p()
    assert L.hg_mel_plan_create(ctypes.byref(plan), 511, 80, 22050, 128, 511, 0.0, 8000.0, None) != 0
    assert b"n_fft must be even" in L.hg_last_error()
    assert L.hg_mel_plan_create(ctypes.byref(plan), 512, 80, 22050, 128, 600, 0.0, 8000.0, None) != 0
    assert b"win_size" in L.hg_last_error()


@pytest.mark.parametrize("case", range(4))
def test_mel_other_shapes_emulation_vs_reference_golden(case):
    """n_fft other than 1024 (SURVEY §8f-4: the reference's Lightning-side callers) runs the direct-DFT kernel;
    its arithmetic, executed on the host, against outputs of the reference's own mel_spectrogram
    (tests/golden/make_golden_mel_other.py)."""
    from test_oracle_cpu import mel_close
    z = load_npz("mel_other.npz")
    n_fft, nm, sr, hop, win, fmin, fmax = [int(v) for v in z["cases"][case]]
    L = _lib.lib()
    plan = ctypes.c_void_p()
    assert L.hg_mel_plan_create(ctypes.byref(plan), n_fft, nm, sr, hop, win, float(fmin), float(fmax), None) == 0
    y = np.ascontiguousarray(z["y"])
    b, t = y.shape
    frames = L.hg_mel_num_frames(plan, t)
    out = np.zeros((b, nm, frames), np.float32)
    assert L.hg_mel_emulate_host(plan, y.ctypes.data, b, t, out.ctypes.data) == 0
    L.hg_mel_plan_destroy(plan)
    ref = z[f"mel_{case}"]
    assert out.shape == ref.shape
    mel_close(out.astype(np.float64), ref, 2e-4)


def test_segment_sampler_draw_rule_matches_reference():
    """MelDataset.__getitem__ draws random.randint(0, len - seg) inclusive (meldataset.py:145-146) and right
    zero-pads short utterances (:150)."""
    import random
    from hifigan_b200.meldataset import SegmentSampler
    s = SegmentSampler.__new__(SegmentSampler)
    s.segment_length, s.lengths, s.offsets, s.rng = 8, [20, 5, 8], [0, 20, 25, 33], random.Random(1234)
    picks = s.draw([0, 1, 2, 0])
    ref = random.Random(1234)
    want = [(0 + ref.randint(0, 12), 8), (20, 5), (25 + ref.randint(0, 0), 8), (0 + ref.randint(0, 12), 8)]
    assert picks == want


def test_segment_sampler_fine_tuning_draw_rule_matches_reference():
    """fine-tuning branch (meldataset.py:163-172): mel_start = random.randint(0, F - fps - 1), audio cropped at
    mel_start * hop; short utterances keep offset 0 and are padded."""
    import random
    from hifigan_b200.meldataset import SegmentSampler
    s = SegmentSampler.__new__(SegmentSampler)
    s.segment_length, s.hop_size, s.frames_per_seg = 8, 2, 4
    s.lengths, s.offsets = [20, 5, 8], [0, 20, 25, 33]
    s.mel_frames, s.mel_offsets = [10, 3, 5], [0, 10, 13, 18]
    s.rng = random.Random(7)
    picks = s.draw_fine_tuning([0, 1, 2, 0])
    ref = random.Random(7)
    m0 = ref.randint(0, 10 - 4 - 1)
    want = [(0 + 2 * m0, 8, 0 + m0, 4), (20, 5, 10, 3)]
    m2 = ref.randint(0, 5 - 4 - 1)
    want.append((25 + 2 * m2, 8, 13 + m2, 4))
    m3 = ref.randint(0, 10 - 4 - 1)
    want.append((0 + 2 * m3, 8, 0 + m3, 4))
    assert picks == want


def test_reference_style_top_level_imports(tmp_path):
    """`src/`-on-PYTHONPATH spelling of the reference (inference.py:9-11) resolves to this package."""
    import subprocess
    import sys
    code = ("from env import AttrDict; from meldataset import mel_spectrogram, MAX_WAV_VALUE, load_wav; "
            "from models import Generator; from utils import get_padding; "
            "import hifigan_b200; assert Generator is hifigan_b200.Generator; print('ok')")
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "hifi-gan_b200", "compat") + os.pathsep + ROOT)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=tmp_path)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr


def test_shipped_configs_match_upstream_values():
    """config_v1/v2/v3.json (deleted by the fork, restated here) carry the keys Generator consumes."""
    for v in ("v1", "v2", "v3"):
        h, ref = H.load_config(v), O.config(v)
        assert all(h[k] == ref[k] for k in ref)
        H.Generator(h)
    assert H.load_config("v3").resblock == "2" and H.load_config("v1").upsample_initial_channel == 512


def test_inference_driver_length_buckets():
    """hifigan_b200.inference: files are sorted by length and stacked into ragged batches whose padding stays below
    max_waste (the kernels take per-item lengths, so stacking never changes anyone's samples); batches are capped;
    max_waste = 0 stacks equal lengths only."""
    from hifigan_b200.inference import bucket_by_length
    items = [("a", torch.zeros(80, 100)), ("b", torch.zeros(80, 70)), ("c", torch.zeros(80, 100)),
             ("d", torch.zeros(80, 96)), ("e", torch.zeros(80, 30))]
    got = [[n for n, _ in b] for b in bucket_by_length(items, 3)]
    assert got == [["e"], ["b", "d", "a"], ["c"]]          # 30 alone (57 % padding with 70), then capped at 3
    got = [[n for n, _ in b] for b in bucket_by_length(items, 8, max_waste=0.0)]
    assert got == [["e"], ["b"], ["d"], ["a", "c"]]
    assert bucket_by_length([], 4) == []


def test_optimizer_state_roundtrip_with_torch_adamw():
    """train_loop.optimizer_state_dict writes torch.optim.AdamW's own state_dict format (UPSTREAM do_* files): a torch
    optimizer loads it, and a state_dict produced BY torch (after two real steps) loads back into the flat buffers."""
    import torch.nn as nn
    from hifigan_b200.train import FlatParams
    from hifigan_b200.train_loop import load_optimizer_state_dict, optimizer_state_dict
    torch.manual_seed(0)
    net = nn.Sequential(nn.Conv1d(3, 4, 3), nn.Conv1d(4, 2, 5))
    params = list(net.parameters())
    opt = torch.optim.AdamW(params, 2e-4, betas=[0.8, 0.99])
    for _ in range(2):
        for p in params:
            p.grad = torch.randn_like(p)
        opt.step()
    ref = opt.state_dict()
    flat = FlatParams(net, "cpu")
    order = list(reversed(params))                      # any order: UPSTREAM's D optimizer is chain(msd, mpd)
    opt2 = torch.optim.AdamW(order, 2e-4, betas=[0.8, 0.99])
    for p in order:
        p.grad = torch.zeros_like(p)
    opt2.step()
    load_optimizer_state_dict(flat, params, ref)
    assert int(flat.step_dev.item()) == 2
    sd = optimizer_state_dict(flat, order, 2e-4, (0.8, 0.99))
    opt2.load_state_dict(sd)                            # torch accepts the format
    for j, p in enumerate(order):
        i = params.index(p) if False else [k for k, q in enumerate(params) if q is p][0]
        assert torch.equal(opt2.state_dict()["state"][j]["exp_avg"], ref["state"][i]["exp_avg"])
        assert torch.equal(opt2.state_dict()["state"][j]["exp_avg_sq"], ref["state"][i]["exp_avg_sq"])
        assert float(opt2.state_dict()["state"][j]["step"]) == 2.0


def test_flat_param_spans_of_the_sub_discriminators_tile_the_buffer():
    """Each sub-discriminator updates its own slice of the flat parameter / gradient / moment buffers on its own lane
    (DiscriminatorTrainer.run_phases): the slices must be contiguous, 16-byte aligned and cover the buffer exactly."""
    from hifigan_b200.train import FlatParams
    mpd, msd = H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator()
    flat = FlatParams(torch.nn.ModuleList([mpd, msd]), "cpu")
    spans = [flat.span_of(d) for d in list(mpd.discriminators) + list(msd.discriminators)]
    assert spans[0][0] == 0 and spans[-1][1] == flat.numel
    assert all(a[1] == b[0] for a, b in zip(spans, spans[1:])) and all(lo % 4 == 0 for lo, _ in spans)
    for d, (lo, hi) in zip(list(mpd.discriminators) + list(msd.discriminators), spans):
        n = sum((p.numel() + 3) // 4 * 4 for p in d.parameters())
        assert hi - lo == n
        for p in d.parameters():                      # every parameter is a view into its slice
            off = (p.data_ptr() - flat.p.data_ptr()) // 4
            assert lo <= off and off + p.numel() <= hi
    with pytest.raises(RuntimeError):
        flat.span_of(torch.nn.ModuleList([mpd.discriminators[0], msd.discriminators[1]]))


@pytest.mark.parametrize("fmax,t", [(None, 8192), (8000, 5000)])
def test_mel_backward_kernel_arithmetic_on_host_vs_autograd(fmax, t):
    """hg_mel_bwd_emulate_host runs the backward kernel's own phase functions (forward FFT, complex un-pack, CSR
    gradient, the Hermitian-packed adjoint transform, window, reflect fold-back) with the threads serialised; checked
    against torch autograd through the fp64 oracle mel, including a silent item (clamp: zero gradient) and the
    reflect-padded edges."""
    L = _lib.lib()
    ya = O.synthetic_audio(3, t, seed=4)
    ya[1] = 0.0                                           # below the 1e-5 clamp everywhere
    g = torch.Generator().manual_seed(1)
    yd = ya.double().requires_grad_(True)
    mel = O.mel_spectrogram(yd, 1024, 80, 22050, 256, 1024, 0, fmax)
    dmel = torch.randn(mel.shape, generator=g, dtype=torch.float64)
    (mel * dmel).sum().backward()
    plan = ctypes.c_void_p()
    assert L.hg_mel_plan_create(ctypes.byref(plan), 1024, 80, 22050, 256, 1024, 0.0, -1.0 if fmax is None else float(fmax),
                                None) == 0
    y32 = np.ascontiguousarray(ya.numpy())
    d32 = np.ascontiguousarray(dmel.float().numpy())
    dy = np.zeros_like(y32)
    assert L.hg_mel_bwd_emulate_host(plan, y32.ctypes.data, d32.ctypes.data, 3, t, dy.ctypes.data) == 0
    L.hg_mel_plan_destroy(plan)
    ref = yd.grad.numpy()
    assert np.all(dy[1] == 0.0) and np.all(ref[1] == 0.0)
    for i in (0, 2):
        err = np.abs(dy[i] - ref[i]).max() / np.abs(ref[i]).max()
        cos = float(np.dot(dy[i], ref[i]) / (np.linalg.norm(dy[i]) * np.linalg.norm(ref[i])))
        assert err < 2e-3 and cos > 0.99999, (i, err, cos)


@pytest.mark.parametrize("workload", ["cfg1", "train"])
def test_bench_reference_arm_contract(workload):
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints ONE JSON line with the contract's
    keys, runs without a GPU, and — under torchrun-style env with RANK != 0 — exits 0 without work."""
    import json
    import subprocess
    import sys
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload, "--steps", "1",
           "--warmup", "0"]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    other = subprocess.run(cmd + ["--gpus", "2"], capture_output=True, text=True, cwd=ROOT, timeout=600, env=env)
    assert other.returncode == 0 and not [l for l in other.stdout.splitlines() if l.startswith("{")]


def test_bench_dump_sample_is_seeded_and_bounded(tmp_path):
    """`bench.py --dump-outputs`: an output above DUMP_ARRAY_BYTES keeps the same whole items, in batch order, on every
    call (the default line's 64 x 262 144-sample waveform -> 16 items); smaller outputs and scalars are kept whole;
    the files hold exactly what was kept, as float32."""
    import bench
    y = torch.randn(64, 1, 262144)
    a, b = bench.dump_sample(y), bench.dump_sample(y.clone())
    assert a.shape == (16, 1, 262144) and a.dtype == torch.float32 and torch.equal(a, b)
    items = [i for i in range(64) if any(torch.equal(y[i], r) for r in a)]
    assert len(items) == 16 and torch.equal(y[items], a)
    small, loss = torch.randn(16, 1, 8192, dtype=torch.float64), torch.tensor(2.5)
    assert torch.equal(bench.dump_sample(small), small.float()) and bench.dump_sample(loss).shape == ()
    bench.write_outputs(str(tmp_path / "out"), {"y_g_hat": a, "loss": bench.dump_sample(loss)})
    assert sorted(os.listdir(tmp_path / "out")) == ["loss.npy", "y_g_hat.npy"]
    got = np.load(tmp_path / "out" / "y_g_hat.npy")
    assert got.dtype == np.float32 and np.array_equal(got, a.numpy())
    assert np.load(tmp_path / "out" / "loss.npy") == np.float32(2.5)


def test_epoch_learning_rate_matches_torch_exponential_lr():
    """train_loop.epoch_learning_rate vs the reference's scheduler (UPSTREAM train.py: ExponentialLR(gamma=h.lr_decay,
    last_epoch=last_epoch), one scheduler.step() per epoch): from scratch, and resumed from a do_* file saved in epoch 2."""
    from hifigan_b200.train_loop import epoch_learning_rate
    h = H.AttrDict(dict(learning_rate=2e-4, lr_decay=0.999, adam_b1=0.8, adam_b2=0.99))
    p = [torch.nn.Parameter(torch.zeros(1))]
    opt = torch.optim.AdamW(p, h.learning_rate, betas=[h.adam_b1, h.adam_b2])
    sch = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=h.lr_decay, last_epoch=-1)
    saved = None
    for epoch in range(5):
        assert opt.param_groups[0]["lr"] == pytest.approx(epoch_learning_rate(h, epoch), rel=1e-12)
        p[0].grad = torch.ones(1)
        opt.step()
        if epoch == 2:
            saved = opt.state_dict()          # what a do_* file written during epoch 2 holds
        sch.step()
    opt2 = torch.optim.AdamW(p, h.learning_rate, betas=[h.adam_b1, h.adam_b2])
    opt2.load_state_dict(saved)
    sch2 = torch.optim.lr_scheduler.ExponentialLR(opt2, gamma=h.lr_decay, last_epoch=2)
    for epoch in range(2, 6):                 # UPSTREAM resumes with `for epoch in range(max(0, last_epoch), ...)`
        assert opt2.param_groups[0]["lr"] == pytest.approx(epoch_learning_rate(h, epoch), rel=1e-12)
        opt2.step()
        sch2.step()


def test_lane_stamps_are_off_unless_asked_for(monkeypatch):
    """TrainStep's time marks launch nothing by default (they would change the step's launch count)."""
    from hifigan_b200.train import LaneStamps
    monkeypatch.delenv("HG_LANE_STAMPS", raising=False)
    st = LaneStamps(torch.device("cpu"))
    st.begin()
    st.mark("start")                        # no-op: would need the CUDA library otherwise
    assert not st.on and st.names == [] and st.read() == {}
