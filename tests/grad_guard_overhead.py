"""Cost of the gradient guard (h.clip_grad_norm) in the graph-replayed training step, one process on one GPU:

    python tests/grad_guard_overhead.py [--rounds 6] [--steps 20] [--batch 16]

V1 at batch 16 x 8192, two TrainSteps with the same seeded weights, one with the guard off and one with it on
(clip_grad_norm = inf: nothing is clipped, the norm and the skip test still run), timed with CUDA events over
`steps` replays per round, alternating for `rounds` rounds.  Then the guard's own kernels alone (the sums of squares
of the G buffer and of the eight D slices, and one finalize), so that the rest of the difference is the lane join.
Prints one JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hifigan_b200 as H                         # noqa: E402
from hifigan_b200.configs import load_config     # noqa: E402
from hifigan_b200.train import TrainStep         # noqa: E402


def events_ms(fn, reps: int) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--batch", type=int, default=16)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    g = torch.Generator().manual_seed(7)
    ya = (0.3 * torch.randn(a.batch, 8192, generator=g)).clamp_(-0.95, 0.95).cuda()
    x = H.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, 8000)
    y_mel = H.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, None)
    steps = {}
    for mode in ("off", "on"):
        h = load_config("v1")
        if mode == "on":
            h.clip_grad_norm = float("inf")
        torch.manual_seed(1234)
        steps[mode] = TrainStep(H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator(), h, "cuda")
        for _ in range(steps[mode].warmup_calls + 3):
            steps[mode].step_graphed(x, ya.unsqueeze(1), y_mel)
    torch.cuda.synchronize()
    times = {"off": [], "on": []}
    for _ in range(a.rounds):
        for mode in ("off", "on"):
            ts = steps[mode]
            times[mode].append(events_ms(lambda: ts.step_graphed(x, ya.unsqueeze(1), y_mel), a.steps))
    on = steps["on"]
    gflat, dflat = on.G.flat, on.D.flat
    norm_g = events_ms(gflat.grad_norm, 50)
    norm_d = events_ms(lambda: [dflat.grad_norm(i, *on.D.spans[i]) for i in range(len(on.D.spans))], 50)
    fin = events_ms(lambda: dflat.finalize_norm(1.0), 50)
    med = {k: statistics.median(v) for k, v in times.items()}
    print(json.dumps({"gpu": smi, "batch": a.batch, "rounds": a.rounds, "steps_per_round": a.steps,
                      "ms_per_step_off": times["off"], "ms_per_step_on": times["on"],
                      "median_off": med["off"], "median_on": med["on"], "median_diff": med["on"] - med["off"],
                      "sumsq_g_ms": norm_g, "sumsq_d_8_slices_serial_ms": norm_d, "finalize_ms": fin,
                      "numel_g": gflat.numel, "numel_d": dflat.numel,
                      "launches_per_step_off": steps["off"].launches_per_step,
                      "launches_per_step_on": on.launches_per_step}), flush=True)


if __name__ == "__main__":
    main()
