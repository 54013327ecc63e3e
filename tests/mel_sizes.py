"""Throughput of the mel front-end per STFT size (n_fft 256 / 512 / 1024 / 2048, hop n_fft / 4, 80 mels), and one
graphed training step of the 44.1 kHz recipe.  Tool, not a pytest module; prints one JSON line per record.

    python tests/mel_sizes.py              # forward + backward per size, then the recipe-A training step
    python tests/mel_sizes.py --no-train   # the mel records only

Per size: 65 536 frames a call (64 items x 1024 frames); at least 4 rotating input / output sets spanning at least
256 MB together (twice the 126 MB L2), so no call finds its input in L2.  Algorithmic bytes:
forward hop x 4 (samples) + num_mels x 4 (output) per frame; backward 2 x hop x 4 (samples read, gradient written)
+ num_mels x 4 (incoming mel gradient) per frame.  The card's name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NUM_MELS, ITEMS, FRAMES_PER_ITEM = 80, 64, 1024
L2_ROTATION = 256 * 2 ** 20          # bytes the rotating input / output sets span at least: twice the 126 MB L2


def emit(rec):
    print(json.dumps(rec), flush=True)


def hbm_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    return 6650.0, "fallback (B200 sustained copy bandwidth, 6.65 TB/s)"


def card():
    rec = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        rec["power_limit_and_max_sm_clock"] = out.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        rec["power_limit_and_max_sm_clock"] = "unknown"
    return rec


def timed(run, n, sets):
    for i in range(sets):
        run(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        run(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def mel_records(peak):
    import hifigan_b200 as H
    from hifigan_b200 import _lib
    L, st = _lib.lib(), torch.cuda.current_stream().cuda_stream
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(7)
    for n_fft in (256, 512, 1024, 2048):
        hop = n_fft // 4
        t = FRAMES_PER_ITEM * hop                               # frames = t // hop with the reflect padding
        args = (n_fft, NUM_MELS, 22050, hop, n_fft, 0, 8000)
        sets = max(4, -(-L2_ROTATION // (ITEMS * (t + NUM_MELS * FRAMES_PER_ITEM) * 4)))
        ys = [torch.rand(ITEMS, t, generator=g, device=dev) * 1.9 - 0.95 for _ in range(sets)]
        H.mel_spectrogram(ys[0][:1], *args)                     # creates / caches the plan
        plan = H.meldataset.torch_mels[f"{ys[0].device}_{n_fft}_{NUM_MELS}_22050_{hop}_{n_fft}_0_8000_False"]
        frames = plan.frames(t)
        nframes = ITEMS * frames
        outs = [torch.empty(ITEMS, NUM_MELS, frames, device=dev) for _ in range(sets)]
        fwd = lambda i: _lib.check(L.hg_mel_fwd(plan.handle, ys[i % sets].data_ptr(), ITEMS, t,
                                                outs[i % sets].data_ptr(), 0, st), "hg_mel_fwd")
        ms = timed(fwd, 40, sets)
        gb = nframes * (hop * 4 + NUM_MELS * 4) / 1e9
        rec = {"record": "mel_fwd", "n_fft": n_fft, "hop": hop, "frames_per_call": nframes, "ms_per_call": ms,
               "frames_per_s": nframes / ms * 1e3, "algorithmic_GBps": gb / ms * 1e3,
               "frac_of_hbm": gb / ms * 1e3 / peak}
        emit(rec)
        dys = [torch.zeros(ITEMS, t, device=dev) for _ in range(sets)]
        bwd = lambda i: _lib.check(L.hg_mel_bwd(plan.handle, ys[i % sets].data_ptr(), outs[i % sets].data_ptr(),
                                                ITEMS, t, dys[i % sets].data_ptr(), st), "hg_mel_bwd")
        try:
            ms = timed(bwd, 20, sets)
        except _lib.HgError as e:                              # a build without a backward at this size
            emit({"record": "mel_bwd", "n_fft": n_fft, "unsupported": str(e)[:200]})
        else:
            gb = nframes * (2 * hop * 4 + NUM_MELS * 4) / 1e9
            emit({"record": "mel_bwd", "n_fft": n_fft, "hop": hop, "frames_per_call": nframes, "ms_per_call": ms,
                  "frames_per_s": nframes / ms * 1e3, "algorithmic_GBps": gb / ms * 1e3,
                  "frac_of_hbm": gb / ms * 1e3 / peak})
        del ys, outs, dys
        torch.cuda.empty_cache()


def train_record(steps=20, warmup=5):
    """one graphed TrainStep of the 44.1 kHz recipe (V1 with upsample_rates [8,8,4,2], n_fft 2048, hop 512),
    batch 16 x 16384 samples"""
    import hifigan_b200 as H
    from hifigan_b200.train import TrainStep
    from oracle import hifigan_oracle as O
    h = dict(O.config("v1"))
    h.update(upsample_rates=[8, 8, 4, 2], upsample_kernel_sizes=[16, 16, 8, 4], n_fft=2048, hop_size=512,
             win_size=2048, sampling_rate=44100, segment_size=16384, fmax=None)
    h = H.AttrDict(h)
    torch.manual_seed(1234)
    ts = TrainStep(H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator(), h, "cuda")
    batches = []
    for i in range(4):
        ya = (torch.rand(16, h.segment_size, generator=torch.Generator().manual_seed(i)) * 1.6 - 0.8).cuda()
        mel = lambda fmax: H.mel_spectrogram(ya, h.n_fft, h.num_mels, h.sampling_rate, h.hop_size, h.win_size, h.fmin,
                                             fmax)
        batches.append((mel(h.fmax), ya.unsqueeze(1), mel(h.fmax_for_loss)))
    for i in range(warmup):
        ts.step_graphed(*batches[i % 4])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        out = ts.step_graphed(*batches[i % 4])
    e1.record()
    torch.cuda.synchronize()
    emit({"record": "train_step_recipe_a", "batch": 16, "segment_size": h.segment_size, "graphed": ts.graph_active,
          "ms_per_step": e0.elapsed_time(e1) / steps, "steps": steps,
          "loss_gen_all": float(out["loss_gen_all"]) if "loss_gen_all" in out else None})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--no-train", action="store_true", help="skip the recipe-A training step")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mel_sizes.py needs a GPU")
    torch.cuda.set_device(0)
    peak, src = hbm_gbs()
    emit(dict(card(), hbm_gbs=peak, hbm_gbs_source=src))
    mel_records(peak)
    if not a.no_train:
        train_record()


if __name__ == "__main__":
    main()
