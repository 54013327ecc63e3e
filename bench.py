#!/usr/bin/env python
"""bench.py — headline benchmark of the hifigan_b200 hot path (contract: see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg1|v3|train]

A "step" is one Generator forward over one batch of synthetic mels.  Default workload = BASELINE.json
configs[1]: V1 Generator, batch 64 x [80 x 1024-frame] mels (16 777 216 output samples per step) per GPU.
For N > 1 (launched by torchrun, one rank per GPU) every rank runs its own batch — inference shards by
utterance with no data-path collective ("weak" scaling) — the timed region is bracketed by a barrier and a
device synchronize on both sides and the reported time is the max over ranks.

Output: ONE JSON line on rank 0.
  value        device-resident throughput (inputs already in HBM), whole job
  e2e          same metric through the public API with HOST buffers: pinned-host mel -> H2D -> Generator ->
               D2H of the waveform inside the timed region
  roofline     tensor-core roofline of the dominant kernels (tcgen05 conv launches, 62 per V1 step)
  cpu_baseline the oracle port (torch CPU fp32, all host threads) on a bounded sample, rank 0, N == 1 only
  train        (default workload only) the second half of BASELINE.json's metric, "V1 train segments/s": a short
               run of the full training step (BASELINE configs[2]: batch 16 x 8192-sample segments per GPU, G + MPD +
               MSD forward/backward, two AdamW updates; gradient all-reduce over NCCL when N > 1)

--workload train makes the training step the primary metric of the line (same keys).

--dump-outputs DIR writes, after the timed steps, what the primary metric's last timed step returned to its caller as
DIR/<name>.npy (float32; rank 0's shard): the Generator workloads' waveform `y_g_hat`; with --workload train the
training step's `y_g_hat` and losses.  An array above DUMP_ARRAY_BYTES keeps a fixed, seeded selection of whole batch
items (DUMP_SEED).  The inputs depend only on the arguments, so two builds can be compared output for output: the
Generator's waveform repeats bit for bit, while the training step's reductions are not bit-reproducible and its
outputs drift apart over the warm-up + --steps AdamW updates (two runs of one build on a B200, 10 timed steps: losses
within 0.6 %, waveform within 3e-3 absolute).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_SAMPLE = {"v1": 2398848, "v3": 175648}  # SURVEY.md §8(d), algorithmic (2 x MAC)
CONV_POST_FLOP_PER_SAMPLE = {"v1": 2 * 32 * 7, "v3": 2 * 32 * 7}  # not a tensor-core launch
WORKLOADS = {
    "cfg2": dict(version="v1", batch=64, frames=1024, name="V1 Generator inference, batch 64 x 80x1024 mels"),
    "cfg1": dict(version="v1", batch=1, frames=256, name="V1 Generator inference, batch 1 x 80x256 mel"),
    "v3": dict(version="v3", batch=64, frames=1024, name="V3 Generator inference, batch 64 x 80x1024 mels"),
}
SR = 22050
TRAIN = dict(version="v1", batch=16, segment=8192,
             name="V1 full training step (G + MPD + MSD, mel-L1/feature/adversarial losses, 2 x AdamW), "
                  "batch 16 x 8192-sample segments per GPU")
# SURVEY.md §8(d): minimal algorithmic work of one step = 3 F_G + 9 F_D MACs per segment, x2 FLOP/MAC
TRAIN_FLOP_PER_SEGMENT = 214.668e9


# ------------------------------------------------------------------------------------------------ helpers
def shard_range(n_items: int, rank: int, world: int):
    """Contiguous [lo, hi) share of n_items for `rank` (inference shards by utterance, no collective)."""
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


DUMP_ARRAY_BYTES = 16 << 20   # the default line's waveform is 64 MiB: 16 of its 64 items
DUMP_SEED = 0


def dump_sample(t: torch.Tensor) -> torch.Tensor:
    """t as float32 on the host; above DUMP_ARRAY_BYTES only a seeded choice of whole items along dim 0, in order."""
    t = t.detach().float()
    if t.dim() > 0 and t.numel() * 4 > DUMP_ARRAY_BYTES:
        keep = max(1, DUMP_ARRAY_BYTES // (t[0].numel() * 4))
        items = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(DUMP_SEED))[:keep].sort().values
        t = t[items.to(t.device)]
    return t.cpu()


def write_outputs(path: str, arrays) -> None:
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), t.numpy())
    total = sum(t.numel() * 4 for t in arrays.values())
    print(f"bench.py: wrote {len(arrays)} arrays ({total / 2**20:.1f} MiB) to {path}", file=sys.stderr)


def _dist_on() -> bool:
    return torch.distributed.is_available() and torch.distributed.is_initialized()


def max_over_ranks(v: float, device="cuda") -> float:
    if not _dist_on():
        return v
    t = torch.tensor([v], dtype=torch.float64, device=device)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(v: float, device="cuda") -> float:
    if not _dist_on():
        return v
    t = torch.tensor([v], dtype=torch.float64, device=device)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM)
    return float(t.item())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"tflops": float(d["bf16_tflops_sustained"]), "hbm_gbs": float(d["hbm_gbs"]),
                "source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"}
    return {"tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md: ~1.4 PF sustained, 6.65 TB/s)"}


# ------------------------------------------------------------------------------------- CPU baseline (oracle)
def measured_traffic(workload: str, n_conv: int):
    """DRAM bytes (read + write) per conv launch, averaged over the step's conv launches, from the committed ncu
    capture of this same workload (profiles/r01_traffic.json; never measured under the timed run).  None when no
    capture of this workload / launch count is on file."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r01_traffic.json")
    try:
        with open(path) as f:
            d = json.load(f)
    except (OSError, ValueError):
        return None
    if d.get("workload") != workload or d.get("conv_launches") != n_conv:
        return None
    return d["per_launch_avg_bytes"]


def _reference_modules():
    """(models, meldataset, env) of the REFERENCE itself from oracle/_ref (built by oracle/build_ref.py in the build
    container, shipped with the snapshot), or None -> the oracle port is timed instead (kind "port")."""
    try:
        from oracle import build_ref
        if build_ref.available():
            return build_ref.load()
    except Exception:  # noqa: BLE001
        pass
    return None


def cpu_generator_baseline(version: str, frames: int, batch: int, steps: int, warmup: int, best_of: bool = False):
    """The reference's CPU implementation of the Generator forward on a bounded sample, all host threads: the
    reference's own src/models.py (oracle/_ref, kind "reference") when it travelled with the snapshot, else the
    oracle port (torch CPU fp32 = the very ops the reference's CPU path runs, kind "port").
    best_of: BASELINE.md / SURVEY §8d cfg1 protocol — report the best of `steps` runs instead of the mean."""
    from oracle import hifigan_oracle as O   # the timed CPU implementation (allowed here: cpu_baseline leg)
    from hifigan_b200.configs import load_config
    h = load_config(version)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = _reference_modules()
    torch.manual_seed(1234)
    if ref is not None:
        models, _, env = ref
        G = models.Generator(env.AttrDict(dict(h))).eval()
        G.remove_weight_norm()                                   # as inference.py:47-48
        run, kind, what = (lambda x: G(x)), "reference", "the reference's own src/models.py Generator (oracle/_ref)"
    else:
        import hifigan_b200 as H
        Gc = H.Generator(H.AttrDict(h))  # parameter container only; never run on the CPU
        Gc.remove_weight_norm()
        sd = {k: v.detach() for k, v in Gc.state_dict().items()}
        run, kind, what = (lambda x: O.generator_forward(sd, h, x)), "port", "fp32 torch-CPU oracle port"
    torch.manual_seed(0)
    x = torch.randn(batch, 80, frames)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            run(x)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    samples = batch * frames * 256
    t = min(times) if best_of else sum(times) / len(times)
    return {"value": samples / t, "unit": "samples/s", "cores": cores, "kind": kind,
            "sample": f"{version} Generator forward on {batch} x 80x{frames} mels per step ({samples} samples), fp32 on "
                      f"the host CPU, {what}, {'best' if best_of else 'mean'} of {len(times)} timed steps after "
                      f"{warmup} warm-up",
            "ms_per_step": t * 1e3, "xrt": samples / t / SR}


# --------------------------------------------------------------------------------------------- training step
def _reference_train_step(ref, h, batch):
    """UPSTREAM train.py's loop body (SURVEY §3.3) over the REFERENCE's own modules and losses, torch autograd +
    torch.optim.AdamW on the CPU — the composition tests/golden/make_golden_train.py pins."""
    import itertools
    from oracle import hifigan_oracle as O
    models, meldataset, env = ref
    hh = env.AttrDict(dict(h))
    torch.manual_seed(1234)
    G, mpd, msd = models.Generator(hh).train(), models.MultiPeriodDiscriminator().train(), models.MultiScaleDiscriminator().train()
    optim_g = torch.optim.AdamW(G.parameters(), hh.learning_rate, betas=[hh.adam_b1, hh.adam_b2])
    optim_d = torch.optim.AdamW(itertools.chain(msd.parameters(), mpd.parameters()), hh.learning_rate,
                                betas=[hh.adam_b1, hh.adam_b2])
    ya = O.synthetic_audio(batch, 8192, seed=3)
    mel = lambda a, fmax: meldataset.mel_spectrogram(a, hh.n_fft, hh.num_mels, hh.sampling_rate, hh.hop_size,
                                                     hh.win_size, hh.fmin, fmax)
    with torch.no_grad():
        x, y_mel = mel(ya, hh.fmax), mel(ya, hh.fmax_for_loss)
    y = ya.unsqueeze(1)
    Fn = torch.nn.functional

    def step():
        y_g_hat = G(x)
        y_g_hat_mel = mel(y_g_hat.squeeze(1), hh.fmax_for_loss)
        optim_d.zero_grad()
        y_df_r, y_df_g, _, _ = mpd(y, y_g_hat.detach())
        loss_disc_f, _, _ = models.discriminator_loss(y_df_r, y_df_g)
        y_ds_r, y_ds_g, _, _ = msd(y, y_g_hat.detach())
        loss_disc_s, _, _ = models.discriminator_loss(y_ds_r, y_ds_g)
        (loss_disc_s + loss_disc_f).backward()
        optim_d.step()
        optim_g.zero_grad()
        loss_mel = Fn.l1_loss(y_mel, y_g_hat_mel) * 45
        _, y_df_g, fmap_f_r, fmap_f_g = mpd(y, y_g_hat)
        _, y_ds_g, fmap_s_r, fmap_s_g = msd(y, y_g_hat)
        loss = (models.generator_loss(y_ds_g)[0] + models.generator_loss(y_df_g)[0]
                + models.feature_loss(fmap_s_r, fmap_s_g) + models.feature_loss(fmap_f_r, fmap_f_g) + loss_mel)
        loss.backward()
        optim_g.step()
    return step


def cpu_train_baseline(batch: int, steps: int, warmup: int):
    """The reference's CPU implementation of the training step on a bounded sample of the training workload: the
    reference's own modules under torch autograd + torch.optim.AdamW (oracle/_ref, kind "reference") when they
    travelled with the snapshot, else the training oracle (kind "port")."""
    from oracle import hifigan_oracle as O          # allowed here: cpu_baseline / --impl reference legs
    from oracle import train_oracle as TO
    from hifigan_b200.configs import load_config
    h = load_config("v1")
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = _reference_modules()
    if ref is not None:
        step, kind, what = _reference_train_step(ref, h, batch), "reference", "the reference's own modules (oracle/_ref)"
    else:
        import hifigan_b200 as H
        torch.manual_seed(1234)
        G, mpd, msd = H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator()  # parameter containers
        sds = [TO.leaf_params({k: v.detach().clone() for k, v in m.state_dict().items()}) for m in (G, mpd, msd)]
        ya = O.synthetic_audio(batch, 8192, seed=3)
        x = O.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, 8000)
        y_mel = O.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, None)
        optims = TO.make_optimizers(*sds, h)
        step = lambda: TO.train_step(*sds, h, x, ya.unsqueeze(1), y_mel, optims=optims)
        kind, what = "port", "fp32 torch-CPU training oracle"
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return {"value": batch / mean, "unit": "segments/s", "cores": cores, "kind": kind,
            "sample": f"V1 full training step on {batch} x 8192-sample segments per step, fp32 on the host CPU, {what}, "
                      f"torch autograd + torch.optim.AdamW, {len(times)} timed steps", "ms_per_step": mean * 1e3}


KERNEL_CLASSES = (
    # (class, substrings of the kernel name): tensor-core implicit GEMMs first, then the bandwidth-bound helpers
    ("conv fwd + dgrad (tcgen05)", ("conv1d_tc_kernel", "conv1d_tc2_kernel", "resblock_pair_kernel")),
    ("wgrad (tcgen05)", ("wgrad_tc_kernel",)),
    ("weight prep (fold / pack / spectral norm; batched job tables)", ("pack_", "fold_weight", "sn_", "prep_batched")),
    ("wgrad finish / weight-norm bwd", ("wgrad_finish", "weight_norm_bwd", "unpack_wgrad")),
    ("cin=1 / cout=1 ends, pooling", ("disc_first", "disc_last", "conv_post", "avgpool", "ncl_to_nlc")),
    ("losses + mel", ("loss_", "l1_sum", "mel_")),
    ("AdamW", ("adamw",)),
    ("bias column sums", ("colsum",)),
    ("NCCL", ("nccl",)),
)


TRACE_REPLAYS = 2


def train_kernel_classes(fn, args3, flop_tensor: float):
    """Per-kernel-class time of ONE training step from a CUPTI kernel trace (torch.profiler) of two graph replays
    taken AFTER the timed region: never a bench value, it only apportions the step.  Serialised kernel time exceeds
    the step time because the step's stream lanes overlap."""
    from torch.profiler import ProfilerActivity, profile as tprofile
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(TRACE_REPLAYS):
            fn(*args3)
        torch.cuda.synchronize()
    agg, other = {c: [0, 0.0] for c, _ in KERNEL_CLASSES}, [0, 0.0]
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name.lower()
        if name.startswith("memcpy") or name.startswith("memset"):
            cls = None
        else:
            cls = next((c for c, keys in KERNEL_CLASSES if any(k in name for k in keys)), None)
        slot = agg[cls] if cls is not None else other
        slot[0] += 1
        slot[1] += e.time_range.elapsed_us()
    total = sum(v[1] for v in agg.values()) + other[1]
    if total <= 0:
        return None
    out = {c: {"launches_per_step": v[0] / 2, "ms_per_step": v[1] / 2e3, "share": v[1] / total}
           for c, v in agg.items() if v[0]}
    out["other (ATen fill / add / copy, memset)"] = {"launches_per_step": other[0] / 2, "ms_per_step": other[1] / 2e3,
                                                      "share": other[1] / total}
    tc_ms = sum(out[c]["ms_per_step"] for c in ("conv fwd + dgrad (tcgen05)", "wgrad (tcgen05)") if c in out)
    peaks = measured_peaks()
    return {"source": "CUPTI trace of 2 graph replays after the timed region (serialised kernel time; lanes overlap)",
            "serialised_ms_per_step": total / 2e3, "classes": out,
            "tensor_core_kernels": {"ms_per_step": tc_ms, "achieved_tflops": flop_tensor / (tc_ms * 1e-3) / 1e12 if tc_ms else None,
                                    "frac_of_peak": (flop_tensor / (tc_ms * 1e-3) / 1e12 / peaks["tflops"]) if tc_ms else None},
            "helper_share": 1.0 - tc_ms / (total / 2e3)}


def measure_mel(dev, steps: int):
    """mel_spectrogram at the 65 536-frame point of BASELINE configs[4]'s sweep (64 x 262 144 samples, n_fft 1024,
    hop 256, 80 mels): kernel launches through the C-ABI, CUDA events on the launching stream.  Four input / output
    sets (268 MB + 84 MB) rotate so no iteration finds its input in the 126 MB L2."""
    import hifigan_b200 as H
    from hifigan_b200 import _lib
    b, t = 64, 262144
    g = torch.Generator().manual_seed(7)
    ys = [(torch.rand(b, t, generator=g) * 1.9 - 0.95).to(dev) for _ in range(4)]
    H.mel_spectrogram(ys[0], 1024, 80, SR, 256, 1024, 0, 8000)           # creates / caches the plan
    plan = H.meldataset.torch_mels[f"{ys[0].device}_1024_80_{SR}_256_1024_0_8000_False"]
    frames = plan.frames(t)
    outs = [torch.empty(b, 80, frames, dtype=torch.float32, device=dev) for _ in range(4)]
    L, st = _lib.lib(), torch.cuda.current_stream().cuda_stream
    run = lambda i: _lib.check(L.hg_mel_fwd(plan.handle, ys[i % 4].data_ptr(), b, t, outs[i % 4].data_ptr(), 0, st))
    for i in range(4):
        run(i)
    torch.cuda.synchronize()
    n = max(8, 4 * steps)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        run(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    peaks = measured_peaks()
    nframes = b * frames
    gbs = nframes * 1344 / (ms * 1e-3) / 1e9                               # SURVEY §8d: 1 344 algorithmic B / frame
    return {"metric": "mel_spectrogram frames/s", "value": nframes / (ms * 1e-3), "unit": "frames/s", "ms_per_call": ms,
            "frames_per_call": nframes, "launches": n,
            "config": {"workload": "mel_spectrogram, 64 x 262144 samples (65 536 frames), n_fft 1024, hop 256, 80 mels, "
                                   "fmax 8000", "l2": "4 rotating input/output sets (352 MB) > 126 MB L2"},
            "roofline": {"bound": "hbm", "kernel": "mel_kernel2", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": gbs / peaks["hbm_gbs"], "algorithmic_bytes_per_frame": 1344, "traffic": None}}


def measure_train(dev, rank, world, steps: int, warmup: int, batch: int = TRAIN["batch"], keep_outputs: bool = False):
    """Time the full training step.  Returns a dict with device-resident and end-to-end numbers (max over ranks);
    keep_outputs: also what the last timed step returned (dump_sample of each tensor) under "outputs"."""
    import hifigan_b200 as H
    from hifigan_b200 import _lib
    from hifigan_b200.configs import load_config
    from hifigan_b200.train import TrainStep
    h = load_config("v1")
    torch.manual_seed(1234)                                   # same replicated initial weights on every rank
    ts = TrainStep(H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator(), h, dev)
    g = torch.Generator().manual_seed(100 + rank)             # every rank its own shard of the global batch
    seg = TRAIN["segment"]
    t_ax = torch.arange(seg, dtype=torch.float32) / SR
    f0 = 80 + 320 * torch.rand(batch, 1, generator=g)
    host_y = (0.5 * torch.sin(2 * torch.pi * f0 * t_ax) + 0.1 * torch.randn(batch, seg, generator=g)).clamp(-0.95, 0.95)
    host_y = host_y.pin_memory()
    y = host_y.to(dev)
    x = H.mel_spectrogram(y, h.n_fft, h.num_mels, h.sampling_rate, h.hop_size, h.win_size, h.fmin, h.fmax)
    y_mel = H.mel_spectrogram(y, h.n_fft, h.num_mels, h.sampling_rate, h.hop_size, h.win_size, h.fmin, h.fmax_for_loss)
    host_x, host_ymel = x.cpu().pin_memory(), y_mel.cpu().pin_memory()
    y3 = y.unsqueeze(1)
    # the whole step (the NCCL all-reduces included when N > 1) replays as one CUDA graph; eager on request
    fn = ts.step if os.environ.get("HG_TRAIN_EAGER") else ts.step_graphed

    def barrier():
        if _dist_on():
            torch.distributed.barrier()
        torch.cuda.synchronize()

    n_warm = max(warmup, 3, ts.warmup_calls + 1)   # data-parallel: the step re-captures once it has timed its lanes
    for _ in range(n_warm):
        fn(x, y3, y_mel)
    barrier()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn(x, y3, y_mel)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    launches = _lib.launch_count() - n0
    # the graph's static outputs: copied before the end-to-end steps below replay into them
    outputs = {k: dump_sample(v) for k, v in out.items()} if keep_outputs else None
    # end to end: the step's three inputs come from pinned host memory, the logged losses go back to the host
    host_loss = torch.empty(2, dtype=torch.float32).pin_memory()
    f0e, f1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0e.record()
    for _ in range(steps):
        xd = host_x.to(dev, non_blocking=True)
        yd = host_y.to(dev, non_blocking=True).unsqueeze(1)
        md = host_ymel.to(dev, non_blocking=True)
        out = fn(xd, yd, md)
        host_loss.copy_(torch.stack([out["loss_gen_all"], out["loss_disc_all"]]), non_blocking=True)
    f1e.record()
    barrier()
    e2e_ms = f0e.elapsed_time(f1e) / steps
    graphed = ts.graph_active
    # a graph replay launches the captured kernels without passing through the C-ABI counter: report the number
    # of library kernels recorded when the step was captured
    per_step = ts.launches_per_step if graphed else launches / steps
    classes = None
    if not os.environ.get("HG_BENCH_NO_TRACE"):
        if rank == 0:
            try:
                # 3 F_G + 9 F_D MACs per segment run on the tensor-core kernels except the Cin = 1 / Cout = 1 ends (< 1 %)
                classes = train_kernel_classes(fn, (x, y3, y_mel), batch * TRAIN_FLOP_PER_SEGMENT)
            except Exception as e:  # noqa: BLE001   (a profiler problem must not cost the measured numbers)
                classes = {"error": f"{type(e).__name__}: {e}"[:200]}
        else:
            for _ in range(TRACE_REPLAYS):   # the step holds the gradient all-reduces: every rank replays it with rank 0
                fn(x, y3, y_mel)
            torch.cuda.synchronize()
    barrier()
    return {"ms": max_over_ranks(ms), "e2e_ms": max_over_ranks(e2e_ms), "batch": batch, "kernel_classes": classes,
            "segments": sum_over_ranks(float(batch)), "launches_per_step": per_step, "graphed": graphed,
            "h2d": (host_x.numel() + host_y.numel() + host_ymel.numel()) * 4, "d2h": 8, "warmup": n_warm,
            "slice_order": list(ts.D.order),
            "losses": [float(v) for v in host_loss.tolist()], "outputs": outputs}


def train_summary(r, world):
    peaks = measured_peaks()
    sps = r["segments"] / (r["ms"] * 1e-3)
    achieved = sps * TRAIN_FLOP_PER_SEGMENT / 1e12 / world      # per GPU
    return {"metric": "V1 train segments/s", "value": sps, "unit": "segments/s", "ms_per_step": r["ms"],
            "per_gpu_batch": r["batch"], "global_batch": int(r["segments"]),
            "e2e": {"value": r["segments"] / (r["e2e_ms"] * 1e-3), "unit": "segments/s", "ms_per_step": r["e2e_ms"],
                    "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"]},
            "cuda_graph": r["graphed"], "kernel_launches_per_step": r["launches_per_step"],
            "parallelism": f"data-parallel x{world}" + (", NCCL all-reduce of the flat G and D gradient buffers"
                                                        if world > 1 else ""),
            "roofline": {"bound": "tensor", "kernel": "whole step (conv fwd / dgrad / wgrad tcgen05 launches + the rest)",
                         "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
                         "frac": achieved / peaks["tflops"], "traffic": None,
                         "algorithmic_flop_per_segment": TRAIN_FLOP_PER_SEGMENT, "peak_source": peaks["source"]},
            "losses_last_step": {"loss_gen_all": r["losses"][0], "loss_disc_all": r["losses"][1]},
            "warmup_steps": r["warmup"], "gradient_slice_order": r["slice_order"],
            "kernel_classes": r.get("kernel_classes")}


def run_train(args, rank, world, local_rank):
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    sampler = ClockSampler(local_rank)
    sampler.start()
    r = measure_train(dev, rank, world, args.steps, args.warmup, args.per_gpu_batch or TRAIN["batch"],
                      keep_outputs=bool(args.dump_outputs) and rank == 0)
    clocks = sampler.stop()
    if rank != 0:
        return
    if args.dump_outputs:
        write_outputs(args.dump_outputs, r["outputs"])
    t = train_summary(r, world)
    line = {"metric": t["metric"], "value": t["value"], "unit": t["unit"], "n_gpus": world, "steps": args.steps,
            "warmup": r["warmup"], "ms_per_step": t["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": TRAIN["name"].replace("batch 16", f"batch {r['batch']}"), "per_gpu_batch": r["batch"],
                       "global_batch": t["global_batch"],
                       "segment_size": TRAIN["segment"], "weights": "random init, seed 1234",
                       "numerics": "bf16 operands / activations / activation gradients, fp32 accumulate, fp32 "
                                   "parameter gradients, master weights and AdamW state",
                       "l2": "one step touches > 1.5 GB of activations, gradients, weights and optimizer state per "
                             "GPU (> 126 MB L2); no flush needed",
                       "cuda_graph": t["cuda_graph"], "parallelism": t["parallelism"],
                       "gradient_slice_order": t["gradient_slice_order"]},
            "clocks": clocks, "e2e": t["e2e"],
            "gpu_launches": int(t["kernel_launches_per_step"] * args.steps), "roofline": t["roofline"],
            "losses_last_step": t["losses_last_step"], "kernel_classes": t["kernel_classes"]}
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_train_baseline(2, 2, 1)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)

# ------------------------------------------------------------------------------------------------- arms
def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores — the reference's own
    modules from oracle/_ref (kind "reference") when that directory travelled with the snapshot, else the oracle
    port (kind "port").  Rank 0 only."""
    if rank != 0:
        return
    if args.workload == "train":
        r = cpu_train_baseline(2, max(1, args.steps), max(0, min(args.warmup, 1)))
        line = {"impl": "reference", "metric": "V1 train segments/s", "value": r["value"], "unit": "segments/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": TRAIN["name"], "sample": r["sample"]},
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": r["value"], "unit": "segments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return
    wl = WORKLOADS[args.workload]
    # a bounded sample of the arm's workload: ONE utterance of the batch at its full length (the batch only repeats
    # the per-utterance work; ~1 s of 16-core CPU time per step for V1 x 1024 frames)
    r = cpu_generator_baseline(wl["version"], wl["frames"], 1, max(1, args.steps), max(0, min(args.warmup, 2)))
    line = {"impl": "reference", "metric": "V1 audio samples/sec" if wl["version"] == "v1" else "V3 audio samples/sec",
            "value": r["value"], "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "xrt_22050": r["xrt"],
            "config": {"workload": wl["name"], "sample": r["sample"]},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_ours(args, rank, world, local_rank):
    import hifigan_b200 as H
    from hifigan_b200 import _lib
    from hifigan_b200.configs import load_config

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — hifigan_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    wl = WORKLOADS[args.workload]
    ver, batch, frames = wl["version"], wl["batch"], wl["frames"]
    h = load_config(ver)
    torch.manual_seed(1234)
    G = H.Generator(h).to(dev).eval()
    G.remove_weight_norm()
    torch.manual_seed(rank)
    host_mel = torch.randn(batch, 80, frames).pin_memory()
    x = host_mel.to(dev)
    samples = batch * frames * 256
    host_out = torch.empty(batch, 1, frames * 256, dtype=torch.float32).pin_memory()
    eng = G._engine(dev)

    def barrier():
        if _dist_on():
            torch.distributed.barrier()
        torch.cuda.synchronize()

    profile_mode = bool(os.environ.get("HG_BENCH_PROFILE"))  # short run for ncu: never a bench value
    n_warm = args.warmup if profile_mode else max(args.warmup, 3)
    with torch.no_grad():
        for _ in range(n_warm):
            eng.forward(x)
        # ---------------- device-resident timing
        conv_ms = []
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        launches0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            y = eng.forward(x, time_convs=True)
            conv_ms.append(eng.last_conv_events)
        e1.record()
        barrier()
        launches = _lib.launch_count() - launches0
        # the engine-owned buffer: copied before the end-to-end calls below write it again
        outputs = {"y_g_hat": dump_sample(y)} if args.dump_outputs and rank == 0 else None
        ms = e0.elapsed_time(e1) / args.steps
        conv_ms = sum(a.elapsed_time(b) for a, b in conv_ms) / args.steps
        # ---------------- end-to-end through the public API with host buffers
        for _ in range(0 if profile_mode else 2):
            host_out.copy_(G(host_mel.to(dev, non_blocking=True)), non_blocking=True)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(0 if profile_mode else args.steps):
            y = G(host_mel.to(dev, non_blocking=True))
            host_out.copy_(y, non_blocking=True)
        f1.record()
        barrier()
        e2e_ms = f0.elapsed_time(f1) / args.steps
        clocks = sampler.stop()

    ms = max_over_ranks(ms)
    e2e_ms = max_over_ranks(e2e_ms)
    total_samples = sum_over_ranks(float(samples))
    mel = None
    if args.workload == "cfg2" and rank == 0 and not profile_mode:
        # the third kernel family north_star names: the fused mel front-end, against the HBM roofline
        try:
            mel = measure_mel(dev, args.steps)
        except Exception as e:  # noqa: BLE001
            mel = {"error": f"{type(e).__name__}: {e}"[:200]}
    train = None
    if args.workload == "cfg2" and not profile_mode and not args.no_train:
        # second half of BASELINE.json's metric: a short run of the full training step on the same GPUs
        del eng, x
        G._drop_engines()
        torch.cuda.empty_cache()
        try:
            train = train_summary(measure_train(dev, rank, world, args.steps, args.warmup), world)
        except Exception as e:  # noqa: BLE001  (the headline number must survive a failure of the secondary one)
            train = {"error": f"{type(e).__name__}: {e}"}
    if rank != 0:
        return
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    peaks = measured_peaks()
    n_conv = launches // args.steps - 2  # every launch of a step except ncl_to_nlc and conv_post
    conv_flops = samples * (FLOP_PER_SAMPLE[ver] - CONV_POST_FLOP_PER_SAMPLE[ver])
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12
    line = {
        "metric": "V1 audio samples/sec" if ver == "v1" else "V3 audio samples/sec",
        "value": total_samples / (ms * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": n_warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "xrt_22050": total_samples / (ms * 1e-3) / SR,
        "config": {"workload": wl["name"], "per_gpu_batch": batch, "frames": frames,
                   "samples_per_step_per_gpu": samples, "weights": "random init, seed 1234, weight_norm folded",
                   "numerics": "bf16 operands + bf16 activations, fp32 accumulate",
                   "l2": "activations per step (>= 1 GB per layer at cfg2) exceed the 126 MB L2; no flush needed"
                   if samples >= (1 << 22) else "small workload: L2-resident by construction (launch-bound case)",
                   "parallelism": f"batch-parallel x{world}, no collective"},
        "clocks": clocks,
        "e2e": {"value": total_samples / (e2e_ms * 1e-3), "unit": "samples/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": host_mel.numel() * 4, "d2h_bytes_per_step": host_out.numel() * 4},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "kernel": "conv1d_tc_kernel + resblock_pair_kernel (tcgen05 implicit GEMM)",
                     "launches_per_step": n_conv,
                     "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
                     "frac": achieved / peaks["tflops"], "traffic": measured_traffic(args.workload, n_conv),
                     "avg_launch_ms": conv_ms / n_conv, "flop_per_launch_avg": conv_flops / n_conv,
                     "peak_source": peaks["source"]},
    }
    if train is not None:
        line["train"] = train
    if mel is not None:
        line["mel"] = mel
    if profile_mode:
        line["invalid"] = "HG_BENCH_PROFILE run (short warm-up, no e2e): not a bench value"
    if world == 1 and not args.no_cpu_baseline and not profile_mode:
        # BASELINE.json configs[0] exactly (SURVEY §8d cfg1): batch 1 x 80x256 mel, fp32 on the CPU, all host threads,
        # best of 5 after 1 warm-up
        cb = cpu_generator_baseline(ver, 256, 1, 5, 1, best_of=True)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line["cpu_baseline"]["xrt_22050"] = cb["xrt"]
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS) + ["train"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step summary of the default line")
    ap.add_argument("--per-gpu-batch", type=int, default=0,
                    help="--workload train: segments per GPU (default 16 = BASELINE configs[2]; configs[3]'s global "
                         "batch 128 is 64 / 32 / 16 at 2 / 4 / 8 GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computed")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.workload == "train":
            run_train(args, rank, world, local_rank)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if _dist_on():
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
