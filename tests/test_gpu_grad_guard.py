"""Gradient-norm clipping and non-finite step skipping inside the training step (h.clip_grad_norm): the norm
kernels, the guarded AdamW flavour, and TrainStep against the reference rule (tests/grad_guard_ref.py: the training
oracle's step with torch.nn.utils.clip_grad_norm_ + `if isfinite(total): optim.step()`)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def H():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import hifigan_b200
    hifigan_b200._lib.lib()
    return hifigan_b200


def _st():
    return torch.cuda.current_stream().cuda_stream


def _norm(L, x, lo, n, max_norm=float("inf"), grad_scale=1.0, step=None, skipped=None):
    """hg_grad_sumsq on x[lo:lo+n] into one slot, then hg_grad_norm_finalize -> (norm, coef, skip) device tensors"""
    from hifigan_b200 import _lib
    slot = L.hg_grad_norm_slot_size()
    ws = torch.full((slot,), float("nan"), dtype=torch.float64, device="cuda")     # the kernel writes the whole slot
    _lib.check(L.hg_grad_sumsq(x.data_ptr() + 4 * lo, n, ws.data_ptr(), _st()), "hg_grad_sumsq")
    norm, coef = torch.empty(1, device="cuda"), torch.empty(1, device="cuda")
    skip = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    _lib.check(L.hg_grad_norm_finalize(ws.data_ptr(), 1, max_norm, grad_scale, norm.data_ptr(), coef.data_ptr(),
                                       skip.data_ptr(), 0 if step is None else step.data_ptr(),
                                       0 if skipped is None else skipped.data_ptr(), _st()), "hg_grad_norm_finalize")
    return norm, coef, skip


def test_grad_norm_kernel_vs_fp64_and_deterministic(H):
    from hifigan_b200 import _lib
    L = _lib.lib()
    gen = torch.Generator(device="cuda").manual_seed(3)
    n_d = 70_727_114                       # about the D flat buffer (282.9 MB); the step's size is checked below too
    x = torch.randn(n_d + 8, generator=gen, device="cuda") * 1e-3
    for n in (1, 3, 4097, n_d):
        for lo in (0, 1, 3):                # 16-byte aligned and not: the same 4-element groups either way
            ref = torch.linalg.vector_norm(x[lo:lo + n].double()).item()
            got = _norm(L, x, lo, n)[0].item()
            assert abs(got - ref) <= 1e-5 * ref, (n, lo, got, ref)
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                again = _norm(L, x, lo, n)[0]
            torch.cuda.current_stream().wait_stream(s)
            assert again.item() == got, (n, lo, again.item(), got)      # bit-identical on another stream
        # the same values at another alignment give the same bits
        y = torch.empty(n + 1, device="cuda")
        y[1:] = x[:n]
        assert _norm(L, y, 1, n)[0].item() == _norm(L, x, 0, n)[0].item()
    # torch's coefficient, the step counter and the skip counter
    step, skipped = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    nrm, coef, skip = _norm(L, x, 0, 4097, max_norm=0.01, grad_scale=0.5, step=step, skipped=skipped)
    ref = 0.5 * torch.linalg.vector_norm(x[:4097].double()).item()
    assert abs(nrm.item() - ref) <= 1e-5 * ref
    want = torch.clamp(torch.tensor(0.01, dtype=torch.float32) / (nrm.cpu() + 1e-6), max=1.0)
    assert coef.cpu().item() == want.item() and skip.item() == 0 and step.item() == 1 and skipped.item() == 0
    assert _norm(L, x, 0, 4097, max_norm=float("inf"))[1].item() == 1.0
    # one NaN or one Inf anywhere: non-finite norm, skip, the skip counter advances and the step counter does not
    for bad in (float("nan"), float("inf"), float("-inf")):
        for pos in (0, 2, 4095, 4096):
            z = x[:4097].clone()
            z[pos] = bad
            nrm, _, skip = _norm(L, z, 0, 4097, step=step, skipped=skipped)
            assert not np.isfinite(nrm.item()) and skip.item() == 1, (bad, pos)
    assert step.item() == 1 and skipped.item() == 12
    # the step's own D buffer size
    mpd, msd = H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator()
    n_real = sum(p.numel() for p in list(mpd.parameters()) + list(msd.parameters()))
    gbuf = torch.randn(n_real, generator=gen, device="cuda")
    ref = torch.linalg.vector_norm(gbuf.double()).item()
    assert abs(_norm(L, gbuf, 0, n_real)[0].item() - ref) <= 1e-5 * ref


def test_guarded_adamw_bits(H):
    from hifigan_b200 import _lib
    L = _lib.lib()
    gen = torch.Generator(device="cuda").manual_seed(4)
    n = 100_003
    p0, g = torch.randn(n, generator=gen, device="cuda"), torch.randn(n, generator=gen, device="cuda")
    m0, v0 = torch.randn(n, generator=gen, device="cuda") * 0.1, torch.rand(n, generator=gen, device="cuda") * 0.01
    lr = torch.tensor([2e-4], device="cuda")
    gs = 0.5

    def plain(scale, step):
        p, m, v = p0.clone(), m0.clone(), v0.clone()
        st = torch.tensor([step], dtype=torch.int32, device="cuda")
        _lib.check(L.hg_adamw_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, 1.0, 0.8, 0.99, 1e-8,
                                   0.01, 0, st.data_ptr(), lr.data_ptr(), scale, _st()))
        return p, m, v

    def guarded(coef, skip, step):
        p, m, v = p0.clone(), m0.clone(), v0.clone()
        st = torch.tensor([step], dtype=torch.int32, device="cuda")
        c = torch.tensor([coef], dtype=torch.float32, device="cuda")
        k = torch.tensor([skip], dtype=torch.int32, device="cuda")
        _lib.check(L.hg_adamw_step_guarded(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, 1.0, 0.8, 0.99,
                                           1e-8, 0.01, st.data_ptr(), lr.data_ptr(), gs, c.data_ptr(), k.data_ptr(),
                                           _st()))
        return (p, m, v), st

    eq = lambda a, b: all(torch.equal(x, y) for x, y in zip(a, b))
    assert eq(guarded(1.0, 0, 3)[0], plain(gs, 3))
    c = 0.3137
    scaled = float(np.float32(gs) * np.float32(c))            # grad_scale * coef rounded to fp32, as the kernel does
    assert eq(guarded(c, 0, 3)[0], plain(scaled, 3))
    assert not eq(guarded(c, 0, 3)[0], plain(gs, 3))
    (p, m, v), st = guarded(c, 1, 3)
    assert eq((p, m, v), (p0, m0, v0)) and st.item() == 3


def _nets(H, clip):
    from oracle import hifigan_oracle as O
    h = H.AttrDict(O.config("v1"))
    if clip is not None:
        h.clip_grad_norm = clip
    torch.manual_seed(1234)
    nets = (H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator())
    sds = [{k: v.detach().clone() for k, v in m.state_dict().items()} for m in nets]
    return h, nets, sds


def _seeded(H, clip):
    from hifigan_b200.train import TrainStep
    h, nets, sds = _nets(H, clip)
    return h, TrainStep(*nets, h, "cuda"), nets, sds


LOSS_KEYS = ("loss_disc_f", "loss_disc_s", "loss_mel", "loss_fm_f", "loss_fm_s", "loss_gen_f", "loss_gen_s")


def _named_moments(flat, net):
    """{parameter name: (m view, v view)} of `net`'s parameters inside `flat`"""
    where = {id(p): i for i, p in enumerate(flat.params)}
    out = {}
    for k, p in net.named_parameters():
        i = where[id(p)]
        o, n = flat.offsets[i], flat.sizes[i]
        out[k] = (flat.m[o:o + n], flat.v[o:o + n])
    return out


def test_guarded_step_vs_oracle_rule(H):
    """V1 at batch 4: the clip limit is half of the smaller unclipped step-1 norm, so both networks clip.  Step 1
    checks the reported norms against torch's totals and the first moments (AdamW's first update is scale-invariant,
    so only m shows the coefficient: ||m|| = (1 - b1) * min(total, max_norm)); then 8 graph-replayed steps follow
    the oracle like the unguarded trajectory test does."""
    from oracle import hifigan_oracle as O
    from oracle import train_oracle as TO
    from grad_guard_ref import guarded_train_step, make_guarded_optimizers
    batches = [O.synthetic_audio(4, 8192, seed=100 + i) for i in range(8)]
    mels = [(O.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, 8000),
             O.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, None)) for ya in batches]
    _, _, sds = _nets(H, None)
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_default_device("cuda")      # the oracle builds its window / filterbank on the default device
    try:
        leaf = lambda: [TO.leaf_params({k: v.detach().clone().cuda() for k, v in sd.items()}) for sd in sds]
        args0 = (mels[0][0].cuda(), batches[0].cuda().unsqueeze(1), mels[0][1].cuda())
        h = H.AttrDict(O.config("v1"))
        sd_free = leaf()
        free = guarded_train_step(*sd_free, h, *args0, optims=make_guarded_optimizers(*sd_free, h, float("inf")))[0]
        max_norm = 0.5 * min(free["grad_norm_g"], free["grad_norm_d"])
        ref_sds = leaf()
        optims = make_guarded_optimizers(*ref_sds, h, max_norm)
        ref = []
        for i, (ya, (x, y_mel)) in enumerate(zip(batches, mels)):
            ref.append(guarded_train_step(*ref_sds, h, x.cuda(), ya.cuda().unsqueeze(1), y_mel.cuda(), optims)[0])
            if i == 0:
                m1 = [{id(p): optims[j].state[p]["exp_avg"].clone() for p in optims[j].param_groups[0]["params"]}
                      for j in range(2)]
    finally:
        torch.set_default_device("cpu")
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    h, ts, (G, mpd, msd), sds0 = _seeded(H, max_norm)
    init = [{k: v.clone() for k, v in sd.items()} for sd in sds0]
    report = {"max_norm": max_norm, "unclipped": (free["grad_norm_g"], free["grad_norm_d"])}
    for i, (ya, (x, y_mel)) in enumerate(zip(batches, mels)):
        out = ts.step_graphed(x.cuda(), ya.cuda().unsqueeze(1), y_mel.cuda())
        for k in LOSS_KEYS:
            got, want = out[k].item(), ref[i][k]
            assert abs(got - want) <= 3e-2 * abs(want) + 1e-4, (i, k, got, want)
        for net, flat in (("g", ts.G.flat), ("d", ts.D.flat)):
            got, want = out[f"grad_norm_{net}"].item(), float(ref[i][f"grad_norm_{net}"])
            report.setdefault(f"grad_norm_{net}", []).append((round(got, 4), round(want, 4)))
            # every step: the in-graph norm is the fp64 norm of the gradient buffer that step left behind
            own = torch.linalg.vector_norm(flat.g.double()).item()
            assert abs(got - own) <= 1e-5 * own, (i, net, got, own)
            assert out[f"skipped_steps_{net}"].item() == 0
            # against torch's totals: step 1 from the same weights; later steps follow two trajectories that drift
            # apart with the bf16 activations (the losses by up to 3e-2, above), so their norms are reported only
            if i == 0:
                assert abs(got - want) <= 2e-2 * want, (i, net, got, want)
        if i > 0:
            continue
        # the coefficient, seen through the first moments: (1 - b1) * max_norm for each network
        assert free["grad_norm_g"] >= 1.5 * max_norm and free["grad_norm_d"] >= 1.5 * max_norm  # unclipped differs
        for j, (flat, nets, sdr) in enumerate(((ts.G.flat, (G,), ref_sds[:1]), (ts.D.flat, (mpd, msd), ref_sds[1:]))):
            mn = flat.m.double().norm().item()
            report[f"m_norm_{'gd'[j]}"] = mn
            assert abs(mn - 0.2 * max_norm) <= 1e-3 * 0.2 * max_norm, (j, mn, 0.2 * max_norm)
            mine, theirs = [], []
            for net, sd in zip(nets, sdr):
                mom = _named_moments(flat, net)
                for k, (m, _) in mom.items():
                    mine.append(m.flatten())
                    theirs.append(m1[j][id(sd[k])].flatten())
            a, b = torch.cat(mine).double(), torch.cat(theirs).double()
            assert abs(a.norm().item() - b.norm().item()) <= 2e-2 * b.norm().item()
            cos = F.cosine_similarity(a, b, dim=0).item()
            report[f"m_cos_{'gd'[j]}"] = cos
            assert cos >= 0.99, (j, cos)
    assert ts.graph_active
    assert ts.G.flat.step_dev.item() == 8 and ts.D.flat.step_dev.item() == 8
    for net, ref_sd, sd0 in zip((G, mpd, msd), ref_sds, init):
        mine = net.state_dict()
        num = den_a = den_b = 0.0
        for k, v in ref_sd.items():
            if not v.requires_grad:
                continue
            da = (mine[k].detach().float().cpu() - sd0[k]).flatten().double()
            db = (v.detach().cpu() - sd0[k]).flatten().double()
            num += float(da @ db); den_a += float(da @ da); den_b += float(db @ db)
        cos = num / (den_a ** 0.5 * den_b ** 0.5 + 1e-30)
        report[f"update_cos_{type(net).__name__}"] = cos
        assert cos >= 0.98, (type(net).__name__, cos)
    print("grad guard vs oracle:", json.dumps(report))


def test_nonfinite_step_is_skipped_inside_the_graph(H):
    from oracle import hifigan_oracle as O
    h, ts, _, _ = _seeded(H, 1.0)
    ya = O.synthetic_audio(2, 8192, seed=21).cuda()
    x = H.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, 8000)
    y_mel = H.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, None)
    for _ in range(3):                                  # eager, capture + replay, replay
        out = ts.step_graphed(x, ya.unsqueeze(1), y_mel)
    torch.cuda.synchronize()
    assert ts.graph_active
    flats = {"g": ts.G.flat, "d": ts.D.flat}
    state = lambda f: [t.clone() for t in (f.p, f.m, f.v, f.step_dev)]
    before = {k: state(f) for k, f in flats.items()}
    skipped0 = {k: f.skipped_dev.item() for k, f in flats.items()}
    bad = ya.clone()
    bad[1, 4000] = float("nan")                          # the real audio: an ordinary numeric input
    out = ts.step_graphed(x, bad.unsqueeze(1), y_mel)
    torch.cuda.synchronize()
    seen = {}
    for k, f in flats.items():
        norm, skipped = out[f"grad_norm_{k}"].item(), out[f"skipped_steps_{k}"].item()
        did_skip = skipped == skipped0[k] + 1
        assert did_skip == (not np.isfinite(norm)), (k, norm, skipped)
        assert skipped in (skipped0[k], skipped0[k] + 1)
        after = state(f)
        if did_skip:
            assert all(torch.equal(a, b) for a, b in zip(before[k], after)), k
        else:
            assert after[3].item() == before[k][3].item() + 1
        seen[k] = (norm, did_skip)
    assert seen["d"][1], "the discriminator must skip a step whose real audio holds a NaN"
    print("NaN step:", seen)
    steps = {k: f.step_dev.item() for k, f in flats.items()}
    out = ts.step_graphed(x, ya.unsqueeze(1), y_mel)
    torch.cuda.synchronize()
    for k in LOSS_KEYS:
        assert np.isfinite(out[k].item()), k
    for k, f in flats.items():
        assert f.step_dev.item() == steps[k] + 1 and np.isfinite(out[f"grad_norm_{k}"].item())


def test_clip_grad_norm_validation(H):
    from oracle import hifigan_oracle as O
    from hifigan_b200.train import TrainStep
    for bad in (0.0, -1.0, float("nan")):
        h = H.AttrDict(O.config("v1"))
        h.clip_grad_norm = bad
        with pytest.raises(ValueError, match="clip_grad_norm"):
            TrainStep(H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator(), h, "cuda")


def test_train_driver_with_clip_grad_norm(H, tmp_path):
    """train_loop with the key set: finite norms and no skips in the returned dict, and the do_* optimizer state still
    loads into torch.optim.AdamW with `step` = applied updates"""
    from scipy.io.wavfile import write
    from hifigan_b200 import train_loop
    cfg = dict(H.load_config("v1"))
    cfg.update(batch_size=2, seed=1234, num_gpus=0, clip_grad_norm=100.0)
    (tmp_path / "config_v1.json").write_text(json.dumps(cfg))
    wavs = tmp_path / "wavs"
    wavs.mkdir()
    from oracle import hifigan_oracle as O
    audio = O.synthetic_audio(5, 12000, seed=9)
    names = [f"utt{i}" for i in range(5)]
    for n, a in zip(names, audio):
        write(wavs / f"{n}.wav", 22050, (a.numpy() * 32767).astype(np.int16))
    (tmp_path / "training.txt").write_text("\n".join(f"{n}|text" for n in names[:4]))
    (tmp_path / "validation.txt").write_text(f"{names[4]}|text")
    cp = tmp_path / "cp"
    argv = ["--input_wavs_dir", str(wavs), "--input_training_file", str(tmp_path / "training.txt"),
            "--input_validation_file", str(tmp_path / "validation.txt"), "--checkpoint_path", str(cp),
            "--config", str(tmp_path / "config_v1.json"), "--stdout_interval", "1", "--checkpoint_interval", "2",
            "--validation_interval", "1000", "--summary_interval", "1", "--training_epochs", "2"]
    r = train_loop.main(argv)
    assert r["final_steps"] == 4
    assert np.isfinite(r["grad_norm_g"]) and np.isfinite(r["grad_norm_d"]) and r["grad_norm_d"] > 0
    assert r["skipped_steps_g"] == 0 and r["skipped_steps_d"] == 0
    do = torch.load(cp / "do_00000002", map_location="cpu")
    assert set(do) == {"mpd", "msd", "optim_g", "optim_d", "steps", "epoch"}
    msd, mpd = H.MultiScaleDiscriminator(), H.MultiPeriodDiscriminator()
    opt = torch.optim.AdamW(list(msd.parameters()) + list(mpd.parameters()), 2e-4, betas=[0.8, 0.99])
    opt.load_state_dict(do["optim_d"])
    assert float(opt.state_dict()["state"][0]["step"]) == 3.0     # three applied D updates before the save


def test_data_parallel_guard_on_hardware(H):
    """torchrun over every GPU of the box (tests/dp_grad_guard.py): identical norms on all ranks, bit-identical
    replicas after 4 guarded graph-replayed steps, and a NaN in one rank's shard makes every rank skip D."""
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if n >= 8 else 4 if n >= 4 else 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tests", "dp_grad_guard.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "guard consistent on all" in res.stdout
