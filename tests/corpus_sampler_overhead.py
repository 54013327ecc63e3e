"""Cost of training from a packed int16 corpus (CorpusSampler) against the in-memory fp32 pool (SegmentSampler), one
process on one GPU:

    python tests/corpus_sampler_overhead.py [--utts 480] [--rounds 3] [--batches 50]

Synthetic 16-bit wav files (2-8 s at 22.05 kHz) in a temporary directory, packed once; the packed file is then in the
page cache (it was just written), so page faults of a cold corpus are not part of these numbers.
1. `batch()` at V1, batch 16 x 8192, peak normalisation, both samplers in alternating rounds: host time per call
   (enqueue only, no synchronize) and time per call on the device's stream (CUDA events around `batches` calls
   issued back to back; the device waits for the host here, so this is close to the host time).
2. `train_loop.main` at V1, batch 16, one epoch per round, with and without --input_corpus in alternating rounds:
   time per step on the device's stream, from CUDA events recorded just before each step's graph replay (the 6th to
   the last step), so that it covers the replay and the next batch's copy, staging and mel calls, plus any time the
   stream waits for the host, and not how far ahead of the device the host runs.
Prints one JSON line with the card's name and power limit.
"""
import argparse
import gc
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch
from scipy.io.wavfile import write

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hifigan_b200 as H                                    # noqa: E402
from hifigan_b200 import corpus as C, train_loop            # noqa: E402
from hifigan_b200.meldataset import CorpusSampler, SegmentSampler, read_filelist   # noqa: E402
from hifigan_b200.train import TrainStep                    # noqa: E402

SR, SEG, BATCH = 22050, 8192, 16


def time_batches(sampler, draws):
    t0 = time.perf_counter()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for ix in draws:
        sampler.batch(ix)
    host = (time.perf_counter() - t0) / len(draws)
    b.record()
    torch.cuda.synchronize()
    return host * 1e3, a.elapsed_time(b) / len(draws)


def train_round(argv, marks):
    marks.clear()
    train_loop.main(argv)
    torch.cuda.synchronize()
    skip = 5
    return marks[skip].elapsed_time(marks[-1]) / (len(marks) - 1 - skip)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=960)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batches", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    tmp = tempfile.mkdtemp(prefix="corpus_overhead_")
    try:
        run(a, smi, tmp)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run(a, smi, tmp):
    wavs = os.path.join(tmp, "wavs")
    os.makedirs(wavs)
    rng = np.random.default_rng(0)
    names = [f"utt{i:05d}" for i in range(a.utts + 1)]
    for n in names:
        length = int(rng.integers(2 * SR, 8 * SR))
        write(os.path.join(wavs, n + ".wav"), SR, (rng.standard_normal(length) * 3000).clip(-32768, 32767).astype(np.int16))
    with open(os.path.join(tmp, "training.txt"), "w") as f:
        f.write("\n".join(f"{n}|text" for n in names[:-1]))
    with open(os.path.join(tmp, "validation.txt"), "w") as f:
        f.write(f"{names[-1]}|text")
    corpus_path = os.path.join(tmp, "train.hgc")
    paths = read_filelist(os.path.join(tmp, "training.txt"), wavs)
    t0 = time.perf_counter()
    C.pack(paths, corpus_path, SR)
    pack_s = time.perf_counter() - t0
    corpus = C.Corpus(corpus_path)

    # 1. batch() of the two samplers
    mel = (1024, 80, 256, 1024, SR, 0, 8000)
    utts = [train_loop.normalize_peak(train_loop.read_wav(p, SR) / H.MAX_WAV_VALUE) for p in paths]
    samplers = {"segment": SegmentSampler(utts, SEG, *mel, fmax_loss=None, seed=1234),
                "corpus": CorpusSampler(corpus, SEG, *mel, fmax_loss=None, seed=1234)}
    draws = [rng.integers(0, a.utts, BATCH).tolist() for _ in range(a.batches)]
    for s in samplers.values():
        time_batches(s, draws[:5])
    host, dev = {k: [] for k in samplers}, {k: [] for k in samplers}
    for _ in range(a.rounds):
        for k, s in samplers.items():
            hms, dms = time_batches(s, draws)
            host[k].append(hms)
            dev[k].append(dms)
    pool_bytes = samplers["segment"].pool.numel() * 4
    del samplers, utts
    gc.collect()
    torch.cuda.empty_cache()

    # 2. train_loop steps per second
    cfg = dict(H.load_config("v1"))
    cfg.update(batch_size=BATCH, num_gpus=0)
    with open(os.path.join(tmp, "config_v1.json"), "w") as f:
        json.dump(cfg, f)
    marks = []
    original = TrainStep.step_graphed

    def marked(self, *args, **kwargs):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append(ev)
        return original(self, *args, **kwargs)

    TrainStep.step_graphed = marked
    step_ms = {"wavs": [], "corpus": []}
    for r in range(a.rounds):
        for arm in ("wavs", "corpus"):
            argv = ["--input_wavs_dir", wavs, "--input_training_file", os.path.join(tmp, "training.txt"),
                    "--input_validation_file", os.path.join(tmp, "validation.txt"),
                    "--checkpoint_path", os.path.join(tmp, f"cp_{arm}_{r}"), "--config", os.path.join(tmp, "config_v1.json"),
                    "--training_epochs", "1", "--stdout_interval", "100000", "--checkpoint_interval", "100000",
                    "--summary_interval", "100000", "--validation_interval", "100000"]
            if arm == "corpus":
                argv += ["--input_corpus", corpus_path]
            step_ms[arm].append(train_round(argv, marks))
            gc.collect()
            torch.cuda.empty_cache()
    TrainStep.step_graphed = original
    med = lambda v: statistics.median(v)
    print(json.dumps({
        "gpu": smi, "utterances": a.utts, "corpus_samples": int(corpus.pcm.size), "corpus_file_bytes":
        os.path.getsize(corpus_path), "fp32_pool_bytes": pool_bytes, "pack_seconds": round(pack_s, 2),
        "batch": [BATCH, SEG], "batches_per_round": a.batches, "rounds": a.rounds,
        "batch_host_ms": host, "batch_device_ms": dev,
        "median_batch_host_ms": {k: med(v) for k, v in host.items()},
        "median_batch_device_ms": {k: med(v) for k, v in dev.items()},
        "train_steps_per_round": a.utts // BATCH, "train_ms_per_step": step_ms,
        "median_train_ms_per_step": {k: med(v) for k, v in step_ms.items()},
        "median_train_steps_per_s": {k: 1e3 / med(v) for k, v in step_ms.items()}}), flush=True)


if __name__ == "__main__":
    main()
