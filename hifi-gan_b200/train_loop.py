"""The UPSTREAM `train.py` driver (jik876/hifi-gan; the fork deleted the file but its README.md:33-39,64-77 still
documents it) on top of `TrainStep` — SURVEY.md §8(f) ranks 2 and 3.

Same command line (`--input_wavs_dir --input_training_file --input_validation_file --checkpoint_path --config
--training_epochs --stdout_interval --checkpoint_interval --summary_interval --validation_interval`), same
checkpoint files and cadence:

    g_{steps:08d}   {'generator': state_dict}
    do_{steps:08d}  {'mpd', 'msd', 'optim_g', 'optim_d', 'steps', 'epoch'}      (reference utils.py:82-101)

`optim_g` / `optim_d` are written in torch.optim.AdamW's own state_dict format, parameter order as UPSTREAM
(`generator.parameters()`, `chain(msd.parameters(), mpd.parameters())`), so published `do_*` files resume here and
files written here load into torch optimizers.  Resume = newest `g_` / `do_` pair in the checkpoint directory
(`scan_checkpoint`), ExponentialLR(gamma = h.lr_decay) stepped per epoch.

What differs from UPSTREAM, deliberately: the DataLoader workers computing mels on the CPU are replaced by the
GPU-resident `SegmentSampler` (the kernels have no CPU path); audio is peak-normalised per utterance to 0.95 (the
UPSTREAM rule — this fork's `[1, L]` call of librosa.util.normalize normalises per SAMPLE, SURVEY §8a row S);
TensorBoard scalars are written only if tensorboard is installed.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import time
from typing import Dict, List

import numpy as np
import torch

from . import _lib
from .env import AttrDict, build_env
from .meldataset import MAX_WAV_VALUE, SegmentSampler, get_dataset_filelist, mel_spectrogram
from .models import Generator, MultiPeriodDiscriminator, MultiScaleDiscriminator
from .train import FlatParams, TrainStep, shard_batch
from .utils import load_checkpoint, save_checkpoint, scan_checkpoint


# ------------------------------------------------------------------------------------- optimizer state <-> torch
def optimizer_state_dict(flat: FlatParams, params: List[torch.nn.Parameter], lr: float, betas, eps: float = 1e-8,
                         weight_decay: float = 0.01) -> dict:
    """The flat AdamW state of `flat` as a torch.optim.AdamW state_dict over `params` (in that order).  `step` is the
    number of updates applied: with clip_grad_norm set, a skipped non-finite step does not count, as in torch."""
    where = {id(p): i for i, p in enumerate(flat.params)}
    step = float(flat.step_dev.item())
    state = {}
    for j, p in enumerate(params):
        i = where[id(p)]
        o, n = flat.offsets[i], flat.sizes[i]
        state[j] = {"step": torch.tensor(step), "exp_avg": flat.m[o:o + n].view(p.shape).clone(),
                    "exp_avg_sq": flat.v[o:o + n].view(p.shape).clone()}
    group = {"lr": lr, "betas": tuple(betas), "eps": eps, "weight_decay": weight_decay, "amsgrad": False,
             "maximize": False, "foreach": None, "capturable": False, "differentiable": False, "fused": None,
             "params": list(range(len(params)))}
    return {"state": state, "param_groups": [group]}


def load_optimizer_state_dict(flat: FlatParams, params: List[torch.nn.Parameter], sd: dict) -> None:
    """Inverse of optimizer_state_dict; accepts state_dicts written by torch.optim.AdamW (published do_* files)."""
    where = {id(p): i for i, p in enumerate(flat.params)}
    step = 0.0
    for j, p in enumerate(params):
        st = sd["state"].get(j)
        if st is None:
            continue
        i = where[id(p)]
        o, n = flat.offsets[i], flat.sizes[i]
        flat.m[o:o + n].copy_(st["exp_avg"].reshape(-1).to(flat.m.device, torch.float32))
        flat.v[o:o + n].copy_(st["exp_avg_sq"].reshape(-1).to(flat.v.device, torch.float32))
        step = max(step, float(st["step"]))
    flat.step_dev.fill_(int(step))


# ------------------------------------------------------------------------------------------------------- data
def read_wav(path: str, sampling_rate: int) -> torch.Tensor:
    """wav file -> fp32 [L] in [-1, 1] (what torchaudio.load(normalize=True) returns, reference meldataset.py:15-17)."""
    from scipy.io.wavfile import read
    sr, data = read(path)
    if sr != sampling_rate:
        raise ValueError("{} SR doesn't match target {} SR".format(sr, sampling_rate))     # meldataset.py:132-134
    data = np.asarray(data)
    if data.ndim > 1:
        data = data[:, 0]
    if data.dtype == np.int16:
        data = data.astype(np.float32) / MAX_WAV_VALUE
    elif data.dtype == np.int32:
        data = data.astype(np.float32) / 2147483648.0
    return torch.from_numpy(data.astype(np.float32))


def normalize_peak(audio: torch.Tensor) -> torch.Tensor:
    """UPSTREAM `normalize(audio) * 0.95`: peak normalisation of the utterance."""
    peak = audio.abs().max()
    return audio / peak * 0.95 if peak > 0 else audio


def normalize_fork(audio: torch.Tensor) -> torch.Tensor:
    """This fork's literal behaviour (`--normalize fork`): meldataset.py:130 calls librosa.util.normalize on a [1, L]
    array, whose default axis=0 normalises every SAMPLE by its own magnitude -> +-0.95 (zeros stay zero)."""
    return torch.sign(audio) * 0.95


# ------------------------------------------------------------------------------------------------------ driver
def epoch_learning_rate(h, epoch: int) -> float:
    """Learning rate of 0-based epoch `epoch`: UPSTREAM's `ExponentialLR(optim, gamma=h.lr_decay, last_epoch=last_epoch)`
    stepped once per epoch.  From scratch that is lr * gamma^epoch; on resume (last_epoch = the saved epoch, the
    optimizer's `initial_lr` restored from the do_* file) torch's closed form gives the same value for the epoch
    that is re-run and the ones after it (tests/test_host_cpu.py checks both against torch's scheduler)."""
    return float(h.learning_rate) * float(h.lr_decay) ** int(epoch)


def train(rank: int, a, h, local_rank: int = None) -> Dict[str, float]:
    """rank = global rank (gradient exchange, batch shard, logging); local_rank = the GPU of this process."""
    world = h.num_gpus if h.num_gpus > 1 else 1
    local_rank = rank if local_rank is None else local_rank
    if world > 1:
        torch.distributed.init_process_group(backend=h.dist_config['dist_backend'], init_method=h.dist_config['dist_url'],
                                             world_size=h.dist_config['world_size'] * h.num_gpus, rank=rank)
    torch.cuda.manual_seed(h.seed)
    device = torch.device('cuda:{:d}'.format(local_rank))
    torch.cuda.set_device(device)
    generator, mpd, msd = Generator(h), MultiPeriodDiscriminator(), MultiScaleDiscriminator()
    if rank == 0:
        os.makedirs(a.checkpoint_path, exist_ok=True)
        print("checkpoints directory : ", a.checkpoint_path)
    cp_g = cp_do = None
    if os.path.isdir(a.checkpoint_path):
        cp_g, cp_do = scan_checkpoint(a.checkpoint_path, 'g_'), scan_checkpoint(a.checkpoint_path, 'do_')
    steps, last_epoch, state_dict_do = 0, -1, None
    if cp_g is not None and cp_do is not None:
        generator.load_state_dict(load_checkpoint(cp_g, 'cpu')['generator'])
        state_dict_do = load_checkpoint(cp_do, 'cpu')
        mpd.load_state_dict(state_dict_do['mpd'])
        msd.load_state_dict(state_dict_do['msd'])
        steps, last_epoch = state_dict_do['steps'] + 1, state_dict_do['epoch']
    ts = TrainStep(generator, mpd, msd, h, device)       # reads h.clip_grad_norm (optional) like every hyper-parameter
    guarded = ts.clip_grad_norm is not None
    g_params = list(generator.parameters())
    d_params = list(msd.parameters()) + list(mpd.parameters())      # UPSTREAM: chain(msd.parameters(), mpd.parameters())
    if state_dict_do is not None:
        load_optimizer_state_dict(ts.G.flat, g_params, state_dict_do['optim_g'])
        load_optimizer_state_dict(ts.D.flat, d_params, state_dict_do['optim_d'])

    training_files, validation_files = get_dataset_filelist(a)
    random.seed(1234)                                                # MelDataset.__init__ (meldataset.py:104-106)
    random.shuffle(training_files)
    # meldataset.py:126-130: `/ MAX_WAV_VALUE` (quirk kept), then peak normalisation unless fine-tuning
    prep = (lambda a_: a_) if a.fine_tuning else (normalize_fork if getattr(a, "normalize", "peak") == "fork"
                                                   else normalize_peak)
    utts = [prep(read_wav(f, h.sampling_rate) / MAX_WAV_VALUE) for f in training_files]
    npy = lambda f: np.load(os.path.join(a.input_mels_dir, os.path.splitext(os.path.split(f)[-1])[0] + '.npy'))
    sampler = SegmentSampler(utts, h.segment_size, h.n_fft, h.num_mels, h.hop_size, h.win_size, h.sampling_rate, h.fmin,
                             h.fmax, h.fmax_for_loss, seed=1234 + steps, device=device,   # a resumed run draws new crops
                             mels=[npy(f) for f in training_files] if a.fine_tuning else None)   # meldataset.py:155-161
    del utts                                    # the sampler holds the pool on the device; drop the host copy
    val = [prep(read_wav(f, h.sampling_rate) / MAX_WAV_VALUE) for f in validation_files] if rank == 0 else []
    val_mels = [torch.from_numpy(npy(f)).float() for f in validation_files] if (rank == 0 and a.fine_tuning) else None
    sw = None
    if rank == 0:
        try:
            from torch.utils.tensorboard import SummaryWriter
            sw = SummaryWriter(os.path.join(a.checkpoint_path, 'logs'))
        except Exception:  # noqa: BLE001
            sw = None
    n_items = len(training_files)
    per_rank = h.batch_size                      # UPSTREAM: batch_size is per GPU (h.batch_size / h.num_gpus upstream of DDP)
    batches_per_epoch = max(1, n_items // (per_rank * world))
    last = {}
    for epoch in range(max(0, last_epoch), a.training_epochs):
        ts.lr = epoch_learning_rate(h, epoch)                        # the captured graph reads it from device memory
        if rank == 0:
            start = time.time()
            print("Epoch: {}".format(epoch + 1))
        order = list(range(n_items))
        random.Random(1234 + epoch).shuffle(order)                   # DistributedSampler.set_epoch equivalent
        for i in range(batches_per_epoch):
            start_b = time.time()
            lo = (i * world) * per_rank
            glob = order[lo:lo + per_rank * world]
            a0, a1 = shard_batch(len(glob), rank, world) if len(glob) % world == 0 else (0, len(glob))
            x, y, y_mel = sampler.batch(glob[a0:a1])
            out = ts.step_graphed(x, y.unsqueeze(1), y_mel)
            if rank == 0:
                if steps % a.stdout_interval == 0:
                    mel_error = out["loss_mel"].item() / 45
                    last = {"steps": steps, "loss_gen_all": out["loss_gen_all"].item(), "mel_error": mel_error}
                    print('Steps : {:d}, Gen Loss Total : {:4.3f}, Mel-Spec. Error : {:4.3f}, s/b : {:4.3f}'.format(
                        steps, last["loss_gen_all"], mel_error, time.time() - start_b))
                    if guarded:
                        last.update(grad_norm_g=out["grad_norm_g"].item(), grad_norm_d=out["grad_norm_d"].item(),
                                    skipped_steps_g=int(out["skipped_steps_g"].item()),
                                    skipped_steps_d=int(out["skipped_steps_d"].item()))
                        skips = '' if not (last["skipped_steps_g"] or last["skipped_steps_d"]) else \
                            ', Skipped Steps G/D : {:d}/{:d}'.format(last["skipped_steps_g"], last["skipped_steps_d"])
                        print('Steps : {:d}, Grad Norm G : {:4.3f}, Grad Norm D : {:4.3f}{}'.format(
                            steps, last["grad_norm_g"], last["grad_norm_d"], skips))
                if steps % a.checkpoint_interval == 0 and steps != 0:
                    save_checkpoint("{}/g_{:08d}".format(a.checkpoint_path, steps), {'generator': generator.state_dict()})
                    save_checkpoint("{}/do_{:08d}".format(a.checkpoint_path, steps),
                                    {'mpd': mpd.state_dict(), 'msd': msd.state_dict(),
                                     'optim_g': optimizer_state_dict(ts.G.flat, g_params, ts.lr, ts.betas),
                                     'optim_d': optimizer_state_dict(ts.D.flat, d_params, ts.lr, ts.betas),
                                     'steps': steps, 'epoch': epoch})
                if sw is not None and steps % a.summary_interval == 0:
                    sw.add_scalar("training/gen_loss_total", out["loss_gen_all"].item(), steps)
                    sw.add_scalar("training/mel_spec_error", out["loss_mel"].item() / 45, steps)
                    if guarded:
                        sw.add_scalar("training/grad_norm_g", out["grad_norm_g"].item(), steps)
                        sw.add_scalar("training/grad_norm_d", out["grad_norm_d"].item(), steps)
                if steps % a.validation_interval == 0 and val:
                    ts.G.invalidate()       # the module API must re-pack: the last AdamW update ran inside the graph
                    last["val_mel_error"] = validate(generator, val, h, device, val_mels)
                    print('Steps : {:d}, Validation Mel-Spec. Error : {:4.3f}'.format(steps, last["val_mel_error"]))
                    if sw is not None:
                        sw.add_scalar("validation/mel_spec_error", last["val_mel_error"], steps)
                    generator.train()
            steps += 1
        if rank == 0:
            print('Time taken for epoch {} is {} sec\n'.format(epoch + 1, int(time.time() - start)))
    last["final_steps"] = steps
    return last


@torch.no_grad()
def validate(generator: Generator, utterances: List[torch.Tensor], h, device, mels=None) -> float:
    """UPSTREAM validation: mean over files of L1(mel(y), mel(G(x))) on whole utterances (split=False), x = mel_in(y)
    or, fine-tuning, the utterance's precomputed mel."""
    generator.eval()
    err = 0.0
    mel = lambda a_, fmax: mel_spectrogram(a_, h.n_fft, h.num_mels, h.sampling_rate, h.hop_size, h.win_size, h.fmin, fmax)
    for i, y in enumerate(utterances):
        y = y.to(device).reshape(1, -1)
        frames = y.shape[1] // h.hop_size
        if mels is not None:
            x = mels[i].to(device).reshape(1, h.num_mels, -1)
            frames = min(frames, x.shape[2])
            x = x[:, :, :frames].contiguous()
        y = y[:, : frames * h.hop_size]
        if mels is None:
            x = mel(y, h.fmax)
        y_g_hat = generator(x)
        err += torch.nn.functional.l1_loss(mel(y, h.fmax_for_loss), mel(y_g_hat.squeeze(1), h.fmax_for_loss)).item()
    return err / max(1, len(utterances))


def main(argv=None) -> Dict[str, float]:
    print('Initializing Training Process..')
    parser = argparse.ArgumentParser()
    parser.add_argument('--group_name', default=None)
    parser.add_argument('--input_wavs_dir', default='LJSpeech-1.1/wavs')
    parser.add_argument('--input_mels_dir', default='ft_dataset')
    parser.add_argument('--input_training_file', default='LJSpeech-1.1/training.txt')
    parser.add_argument('--input_validation_file', default='LJSpeech-1.1/validation.txt')
    parser.add_argument('--checkpoint_path', default='cp_hifigan')
    parser.add_argument('--config', default='')
    parser.add_argument('--training_epochs', default=3100, type=int)
    parser.add_argument('--stdout_interval', default=5, type=int)
    parser.add_argument('--checkpoint_interval', default=5000, type=int)
    parser.add_argument('--summary_interval', default=100, type=int)
    parser.add_argument('--validation_interval', default=1000, type=int)
    parser.add_argument('--fine_tuning', default=False, type=bool)
    parser.add_argument('--normalize', default='peak', choices=['peak', 'fork'])   # see normalize_fork
    a = parser.parse_args(argv)
    with open(a.config) as f:
        h = AttrDict(json.loads(f.read()))
    build_env(a.config, 'config.json', a.checkpoint_path)
    torch.manual_seed(h.seed)
    if not torch.cuda.is_available():
        raise RuntimeError("hifigan_b200 has no CPU path: a B200 is required")
    h.num_gpus = int(os.environ.get("WORLD_SIZE", "1"))          # one process per GPU, launched by torchrun
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    rank = int(os.environ.get("RANK", str(local_rank)))          # global rank: differs from LOCAL_RANK across nodes
    if h.num_gpus > 1:
        h.dist_config = dict(h.get("dist_config", {}), dist_backend="nccl", dist_url="env://", world_size=1)
        h.batch_size = int(h.batch_size / h.num_gpus)            # UPSTREAM: the configured batch is global
        print('Batch size per GPU :', h.batch_size)
    return train(rank, a, h, local_rank)


if __name__ == '__main__':
    main()
