"""Data-parallel gradient guard (h.clip_grad_norm) on real GPUs:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29547 tests/dp_grad_guard.py

Every rank builds the same seeded networks with the guard on and trains on its shard of a global batch.  Checks that
the reported norms are identical on all ranks (they are computed from the all-reduced gradient bits), that the
replicas stay bit-identical through 4 guarded graph-replayed steps, and that a NaN in ONE rank's shard makes every
rank skip the discriminator update (the all-reduce spreads it).  Tool, not a pytest module (tests/test_gpu_grad_guard.py
launches it); exit code 1 on failure.
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hifigan_b200 as H                         # noqa: E402
from hifigan_b200.configs import load_config     # noqa: E402
from hifigan_b200.train import TrainStep, shard_batch   # noqa: E402


def same_on_all(t: torch.Tensor) -> bool:
    ref = t.clone()
    dist.broadcast(ref, 0)
    flag = torch.tensor([1 if torch.equal(t, ref) else 0], device=t.device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item())


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl")
    dev = torch.device("cuda", local)
    h = load_config("v1")
    h.clip_grad_norm = 1.0
    torch.manual_seed(1234)
    ts = TrainStep(H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator(), h, dev)
    per = 2
    gb = per * world
    g = torch.Generator().manual_seed(5)
    t = torch.arange(8192, dtype=torch.float32)
    f0 = 100.0 + 300.0 * torch.rand(gb, 1, generator=g)
    ya = (0.5 * torch.sin(2 * torch.pi * f0 * t / 22050) + 0.1 * torch.randn(gb, 8192, generator=g)).clamp_(-0.95, 0.95).to(dev)
    mel = lambda a, fmax: H.mel_spectrogram(a, 1024, 80, 22050, 256, 1024, 0, fmax)
    x, y_mel = mel(ya, 8000), mel(ya, None)
    lo, hi = shard_batch(gb, rank, world)
    ok = True
    for _ in range(ts.warmup_calls + 4):
        out = ts.step_graphed(x[lo:hi], ya[lo:hi].unsqueeze(1), y_mel[lo:hi])
        for k in ("grad_norm_g", "grad_norm_d"):
            same = same_on_all(out[k].reshape(1).clone())
            ok = ok and same and bool(torch.isfinite(out[k]).item())
    torch.cuda.synchronize()
    for flat, name in ((ts.G.flat, "G"), (ts.D.flat, "D")):
        same = same_on_all(flat.p) and same_on_all(flat.m) and same_on_all(flat.step_dev)
        if rank == 0:
            print(f"{name}: norms identical and replicas bit-identical after guarded graph-replayed steps: {same}",
                  flush=True)
        ok = ok and same
    # a NaN in rank 0's shard only
    d_before = [t_.clone() for t_ in (ts.D.flat.p, ts.D.flat.m, ts.D.flat.v, ts.D.flat.step_dev)]
    skipped0 = ts.D.flat.skipped_dev.item()
    bad = ya[lo:hi].clone()
    if rank == 0:
        bad[0, 1234] = float("nan")
    out = ts.step_graphed(x[lo:hi], bad.unsqueeze(1), y_mel[lo:hi])
    torch.cuda.synchronize()
    skipped = out["skipped_steps_d"].item() == skipped0 + 1
    kept = all(torch.equal(a, b) for a, b in zip(d_before, (ts.D.flat.p, ts.D.flat.m, ts.D.flat.v, ts.D.flat.step_dev)))
    flag = torch.tensor([1 if (skipped and kept) else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"NaN on rank 0 only: every rank skipped the D update: {bool(flag.item())}", flush=True)
    ok = ok and bool(flag.item()) and same_on_all(ts.G.flat.p) and same_on_all(ts.D.flat.p)
    if rank == 0 and ok:
        print(f"guard consistent on all {world} ranks", flush=True)
    # see tests/dp_check.py: leave without tearing down process groups used inside a CUDA graph
    torch.cuda.synchronize()
    sys.stdout.flush()
    os._exit(0 if ok else 1)


if __name__ == "__main__":
    main()
