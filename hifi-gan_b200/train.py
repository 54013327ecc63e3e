"""The UPSTREAM training step (jik876/hifi-gan train.py; the fork deleted the file but ships every function it
calls — SURVEY.md §3.3) on hand-written sm_100a kernels: forward, backward, AdamW and the data-parallel gradient
all-reduce.  No torch autograd runs here: every gradient is produced by a kernel of libhifigan_b200.so
(include/hifigan_b200.h, "Training step" section) and the chain rule is spelled out below.

    y_g_hat = G(x);  y_g_hat_mel = mel(y_g_hat)
    D step:  loss_disc = sum_d [mean((1 - d(y))^2) + mean(d(y_g_hat.detach())^2)]   over MPD + MSD; AdamW(D)
    G step:  loss_gen  = 45 * L1(y_mel, y_g_hat_mel) + sum_d [2 * sum_l mean|fmap_r - fmap_g| + mean((1 - d(y_g_hat))^2)]
             back through the UPDATED discriminators into G; AdamW(G)

Numerics (declared): bf16 operands and bf16-stored activations / activation gradients, fp32 accumulation,
fp32 parameter gradients, fp32 master weights and optimizer state.
"""
from __future__ import annotations

import os
from ctypes import byref, c_int
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib
from .meldataset import mel_spectrogram, torch_mels
from .models import (LRELU_SLOPE, DiscriminatorP, DiscriminatorS, Generator, MultiPeriodDiscriminator,
                     MultiScaleDiscriminator, ResBlock1, _DiscLayer, _PackedConv, _avgpool, _conv, _device_mean,
                     _g_v, _pad_ch, _round_up, _stream, discriminator_loss, feature_loss, generator_loss)


def _p(x) -> int:
    """device pointer of a tensor / raw int pointer / None"""
    if x is None:
        return 0
    if isinstance(x, int):
        return x
    return x.data_ptr()


def step_losses(generator, mpd, msd, x: torch.Tensor, y: torch.Tensor, y_mel: torch.Tensor, h) -> Dict[str, torch.Tensor]:
    """One training step's loss values, call for call as the reference computes them (no optimizer update):
    the forward half of `TrainStep.step`, through the public module API.  msd is evaluated twice, so a
    train-mode spectral-norm scale advances 4 power iterations per step exactly like the reference."""
    with torch.no_grad():
        y_g_hat = generator(x).clone()
        y_g_hat_mel = mel_spectrogram(y_g_hat.squeeze(1), h.n_fft, h.num_mels, h.sampling_rate, h.hop_size,
                                      h.win_size, h.fmin, h.fmax_for_loss)
        y_df_r, y_df_g, _, _ = mpd(y, y_g_hat)
        loss_disc_f, _, _ = discriminator_loss(y_df_r, y_df_g)
        y_ds_r, y_ds_g, _, _ = msd(y, y_g_hat)
        loss_disc_s, _, _ = discriminator_loss(y_ds_r, y_ds_g)
        loss_mel = _device_mean(y_mel, y_g_hat_mel, 0, 0.0) * 45
        _, y_df_g, fmap_f_r, fmap_f_g = mpd(y, y_g_hat)
        _, y_ds_g, fmap_s_r, fmap_s_g = msd(y, y_g_hat)
        out = {"y_g_hat": y_g_hat, "loss_disc_f": loss_disc_f, "loss_disc_s": loss_disc_s, "loss_mel": loss_mel,
               "loss_fm_f": feature_loss(fmap_f_r, fmap_f_g), "loss_fm_s": feature_loss(fmap_s_r, fmap_s_g),
               "loss_gen_f": generator_loss(y_df_g)[0], "loss_gen_s": generator_loss(y_ds_g)[0]}
        out["loss_disc_all"] = out["loss_disc_s"] + out["loss_disc_f"]
        out["loss_gen_all"] = (out["loss_gen_s"] + out["loss_gen_f"] + out["loss_fm_s"] + out["loss_fm_f"]
                               + out["loss_mel"])
    return out


# ------------------------------------------------------------------------------------------------ flat params
class FlatParams:
    """All parameters of a module re-pointed into ONE fp32 buffer (plus flat gradient and AdamW state buffers):
    the optimizer step is one kernel launch and the data-parallel all-reduce one NCCL call per network.
    state_dict() / load_state_dict() keep working — they copy through the views."""

    def __init__(self, module: nn.Module, device, bind: bool = True):
        """bind=False (the autograd path): only the flat GRADIENT buffer is created; parameters, `.grad` and the
        optimizer state stay torch's."""
        self.module = module
        self.bound = bind
        ps = [p for p in module.parameters()]
        self.sizes = [p.numel() for p in ps]
        # 16-byte aligned offsets so kernels may use vector accesses on any view
        self.offsets, off = [], 0
        for s in self.sizes:
            self.offsets.append(off)
            off += (s + 3) // 4 * 4
        self.numel = off
        self.g = torch.zeros(off, dtype=torch.float32, device=device)
        self.params = ps
        self._grads = {id(p): self.g[o:o + s].view(p.shape) for p, o, s in zip(ps, self.offsets, self.sizes)}
        if not bind:
            for p in ps:
                if p.device != self.g.device or p.dtype != torch.float32 or not p.is_contiguous():
                    raise RuntimeError("hifigan_b200: parameters must be contiguous fp32 tensors on the CUDA device")
            return
        self.p = torch.zeros(off, dtype=torch.float32, device=device)
        self.m = torch.zeros(off, dtype=torch.float32, device=device)
        self.v = torch.zeros(off, dtype=torch.float32, device=device)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=device)   # AdamW step counter (graph-capturable)
        self.lr_dev = torch.zeros(1, dtype=torch.float32, device=device)   # learning rate, read by the kernel
        self._lr_host = None
        self.max_norm: Optional[float] = None          # clip_grad_norm (enable_guard); None: the unguarded update
        with torch.no_grad():
            for p, o, s in zip(ps, self.offsets, self.sizes):
                view = self.p[o:o + s].view(p.shape)
                view.copy_(p.detach().to(device=device, dtype=torch.float32))
                p.data = view
                p.grad = self._grads[id(p)]

    def grad(self, param: torch.Tensor) -> torch.Tensor:
        """the view of the flat gradient buffer the library writes `param`'s gradient into (bound as `param.grad`
        when bind=True; the autograd path keeps it private and hands copies to torch)"""
        return self._grads[id(param)]

    def adamw(self, lr: float, betas=(0.8, 0.99), eps: float = 1e-8, weight_decay: float = 0.01,
              grad_scale: float = 1.0) -> None:
        """torch.optim.AdamW(lr, betas) semantics (UPSTREAM train.py: AdamW(h.learning_rate, [adam_b1, adam_b2])).
        Guarded (enable_guard): after grad_norm and finalize_norm, which advance the step counter themselves."""
        if not self.guarded:
            self.step_dev.add_(1)
        self._adamw(0, self.numel, lr, betas, eps, weight_decay, grad_scale)

    def bump_step(self) -> None:
        """advance the device-side AdamW step counter once per optimizer step (before any adamw_slice of that step)"""
        self.step_dev.add_(1)

    def adamw_slice(self, lo: int, hi: int, lr: float, betas=(0.8, 0.99), eps: float = 1e-8,
                    weight_decay: float = 0.01, grad_scale: float = 1.0) -> None:
        """the same update on elements [lo, hi) of the flat buffers only (after bump_step, or guarded after
        finalize_norm): lets independent parts of a network update on their own stream lanes as soon as their
        gradients are complete"""
        self._adamw(lo, hi, lr, betas, eps, weight_decay, grad_scale)

    def _adamw(self, lo: int, hi: int, lr: float, betas, eps: float, weight_decay: float, grad_scale: float) -> None:
        L, o = _lib.lib(), 4 * lo
        ptrs = (self.p.data_ptr() + o, self.g.data_ptr() + o, self.m.data_ptr() + o, self.v.data_ptr() + o, hi - lo,
                lr, betas[0], betas[1], eps, weight_decay)
        if self.guarded:
            _lib.check(L.hg_adamw_step_guarded(*ptrs, self.step_dev.data_ptr(), self.lr_dev.data_ptr(), grad_scale,
                                               self.clip_coef.data_ptr(), self.skip_flag.data_ptr(), _stream()),
                       "hg_adamw_step_guarded")
        else:
            _lib.check(L.hg_adamw_step(*ptrs, 0, self.step_dev.data_ptr(), self.lr_dev.data_ptr(), grad_scale,
                                       _stream()), "hg_adamw_step")

    # ---- clip_grad_norm_ + skip of non-finite steps (the fork's manual-optimisation callback), inside the graph
    @property
    def guarded(self) -> bool:
        return self.max_norm is not None

    def enable_guard(self, max_norm: float, slots: int = 1) -> None:
        """From now on every update of this network follows
            total = clip_grad_norm_(params, max_norm);  if isfinite(total): optim.step()
        grad_norm() fills `slots` partial sums (one per independently finished part of the buffer), finalize_norm()
        decides, and adamw / adamw_slice read its coefficient and skip flag from device memory.  The results live in
        static device buffers: grad_norm_dev (pre-clip norm, fp32), skipped_dev (int32, cumulative skipped steps)."""
        max_norm = float(max_norm)
        if not max_norm > 0.0:
            raise ValueError(f"clip_grad_norm must be a positive number or inf, got {max_norm}")
        dev = self.p.device
        self.max_norm = max_norm
        self.norm_slots = slots
        self.norm_ws = torch.zeros(slots * _lib.lib().hg_grad_norm_slot_size(), dtype=torch.float64, device=dev)
        self.grad_norm_dev = torch.zeros(1, dtype=torch.float32, device=dev)
        self.clip_coef = torch.ones(1, dtype=torch.float32, device=dev)
        self.skip_flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self.skipped_dev = torch.zeros(1, dtype=torch.int32, device=dev)

    def grad_norm(self, slot: int = 0, lo: int = 0, hi: Optional[int] = None) -> None:
        """sum of squares of gradient elements [lo, hi) into partial-sum slot `slot` (on the current stream)"""
        hi = self.numel if hi is None else hi
        ws = self.norm_ws.data_ptr() + 8 * slot * _lib.lib().hg_grad_norm_slot_size()
        _lib.check(_lib.lib().hg_grad_sumsq(self.g.data_ptr() + 4 * lo, hi - lo, ws, _stream()), "hg_grad_sumsq")

    def finalize_norm(self, grad_scale: float = 1.0) -> None:
        """after every slot is written: the norm of grad_scale * g, the clip coefficient, the skip flag; advances
        step_dev for an applied step and skipped_dev for a skipped one"""
        _lib.check(_lib.lib().hg_grad_norm_finalize(
            self.norm_ws.data_ptr(), self.norm_slots, self.max_norm, grad_scale, self.grad_norm_dev.data_ptr(),
            self.clip_coef.data_ptr(), self.skip_flag.data_ptr(), self.step_dev.data_ptr(),
            self.skipped_dev.data_ptr(), _stream()), "hg_grad_norm_finalize")

    def span_of(self, module: nn.Module) -> Tuple[int, int]:
        """[lo, hi) of the flat buffers covered by `module`'s parameters (they must be contiguous in the buffer)"""
        ids = {id(q) for q in module.parameters()}
        idx = [i for i, q in enumerate(self.params) if id(q) in ids]
        if not idx or idx != list(range(idx[0], idx[-1] + 1)):
            raise RuntimeError("FlatParams.span_of: the module's parameters are not one contiguous run")
        lo = self.offsets[idx[0]]
        hi = self.offsets[idx[-1] + 1] if idx[-1] + 1 < len(self.params) else self.numel
        return lo, hi

    def set_lr(self, lr: float) -> None:
        """the learning rate lives in device memory so that a captured step follows a schedule without re-capture;
        call OUTSIDE graph capture (TrainStep does, before every step)"""
        if lr != self._lr_host:
            self.lr_dev.fill_(lr)
            self._lr_host = lr


class _Lanes:
    """A set of side streams for independent kernel chains (the eight sub-discriminators, the MRF branches, the
    weight-gradient launches beside the data-gradient chain).  fork() makes every lane wait for the work already
    queued on the current stream, join() makes the current stream wait for every lane; both are event waits, so
    under CUDA-graph capture the lanes become parallel branches of the graph."""

    def __init__(self, n: int, device, priorities=None):
        """priorities[i]: CUDA stream priority of lane i (-1 = high, 0 = default / low).  The chains a step waits for
        (forward, data gradients) run on high-priority lanes, parameter-gradient and packing work on low-priority
        ones: when both have thread blocks pending, the critical chain's blocks are placed first.  Captured into the
        step's CUDA graph as kernel-node priorities."""
        pr = priorities if priorities is not None else [0] * n
        self.streams = ([torch.cuda.Stream(device=device, priority=pr[i]) for i in range(n)]
                        if torch.cuda.is_available() else [])

    def fork(self) -> None:
        main = torch.cuda.current_stream()
        for s in self.streams:
            s.wait_stream(main)

    def join(self) -> None:
        main = torch.cuda.current_stream()
        for s in self.streams:
            main.wait_stream(s)

    def lane(self, i: int):
        return torch.cuda.stream(self.streams[i % len(self.streams)])


class LaneStamps:
    """Time marks inside the (graph-replayed) step: hg_timestamp launches on the lanes, read back after the replay.
    On with HG_LANE_STAMPS=1 (tests/lane_stamps.py) or while TrainStep calibrates the order of the gradient slices
    (`force`); otherwise mark() is a no-op and nothing is launched."""

    def __init__(self, device, slots: int = 96):
        self.device, self.slots = device, slots
        self.env_on = bool(os.environ.get("HG_LANE_STAMPS"))
        self.force = False
        self.names: List[str] = []
        self.buf: Optional[torch.Tensor] = None

    @property
    def on(self) -> bool:
        return self.env_on or self.force

    def begin(self) -> None:
        self.names = []                 # the step issues its marks in the same order every time it runs or is captured
        if self.on and self.buf is None:
            self.buf = torch.zeros(self.slots, dtype=torch.int64, device=self.device)

    def mark(self, name: str) -> None:
        if not self.on or self.buf is None or len(self.names) >= self.slots:
            return
        _lib.check(_lib.lib().hg_timestamp(self.buf.data_ptr() + 8 * len(self.names), _stream()), "hg_timestamp")
        self.names.append(name)

    def read(self) -> Dict[str, float]:
        """microseconds since the step's first mark, by name (after a synchronize)"""
        if self.buf is None or not self.names:
            return {}
        v = self.buf[: len(self.names)].cpu().tolist()
        return {n: (t - v[0]) / 1e3 for n, t in zip(self.names, v)}


def allreduce_gradients(flat: FlatParams, group=None, span: Optional[Tuple[int, int]] = None) -> float:
    """Data-parallel exchange step: SUM all-reduce of one network's flat gradient buffer (or of elements [lo, hi) of it)
    over the process group (NCCL over NVLink on the GPUs; gloo in the CPU tests).  Returns the factor the optimizer
    must apply to the summed gradients (1 / world size) — the same averaging DistributedDataParallel performs for the
    reference.  Every rank must issue these calls in the same order; NCCL runs them in that order on its own stream,
    after the work already queued on the CALLER's current stream, and the caller's stream then waits for the result —
    so slices issued from different lanes overlap with the lanes still computing."""
    if not (torch.distributed.is_available() and torch.distributed.is_initialized()):
        return 1.0
    world = torch.distributed.get_world_size(group)
    if world > 1:
        g = flat.g if span is None else flat.g[span[0]:span[1]]
        torch.distributed.all_reduce(g, op=torch.distributed.ReduceOp.SUM, group=group)
    return 1.0 / world


def shard_batch(global_batch: int, rank: int, world: int) -> Tuple[int, int]:
    """[lo, hi) rows of the global batch owned by `rank` (BASELINE configs[3]: global batch 128 over 2/4/8 GPUs)."""
    if global_batch % world:
        raise ValueError(f"global batch {global_batch} does not divide over {world} ranks")
    per = global_batch // world
    return rank * per, (rank + 1) * per


# ------------------------------------------------------------------------------------------------ generator
class _GenLayerGrad:
    """Backward-side state of one packed Generator conv: dgrad filter bank, packed fp32 weight gradient (a view
    into the trainer's flat buffer, zeroed once per backward), and the route back to the weight_norm parameters.
    Every kernel here ACCUMULATES: GeneratorTrainer.backward zeroes the flat packed-gradient buffer and the flat
    parameter-gradient buffer first, so no per-layer memset / copy nodes are needed."""

    def __init__(self, pc: _PackedConv, device, flat: FlatParams, need_dgrad: bool = True):
        self.pc, self.flat = pc, flat
        rows = pc.w.shape[1]
        self.rows = rows
        self.wd = torch.empty(pc.taps, pc.cin_p, rows, dtype=torch.bfloat16, device=device) if need_dgrad else None
        self.dwp_numel = pc.taps * rows * pc.cin_p
        self.dwp = None                                   # assigned by GeneratorTrainer (view into one flat buffer)
        self.db = None                                    # padded bias gradient, only when cout_p != cout
        self.dgrad_pad = (pc.taps - 1) * pc.dil - pc.pad_left

    def pack(self, L) -> None:
        if self.wd is not None:
            pc = self.pc
            _lib.check(L.hg_pack_dgrad_weight(pc.w.data_ptr(), pc.taps, self.rows, pc.cin_p, self.wd.data_ptr(),
                                              _stream()), "hg_pack_dgrad_weight")

    def add_jobs(self, table, finish: str = "finish") -> None:
        """this layer's share of the trainer's batched launches: phase "dgrad" = the data-gradient filter bank (tap
        flip + transpose of the forward bank), phase `finish` = packed dW -> parameter gradients (unpack +
        weight_norm backward, accumulating)"""
        from . import batched
        pc = self.pc
        if self.wd is not None:
            tc, tn = (pc.cin_p + 31) // 32, (self.rows + 31) // 32
            table.add("dgrad", batched.TRANSPOSE_TILE, pc.taps * tc * tn, 32 * 34 * 2, pc.w, dst0=self.wd,
                      ints=(pc.taps, self.rows, pc.cin_p, tc, tn))
        m = pc.module
        g, v = _g_v(m)
        dv, dg = self.flat.grad(v), None if g is None else self.flat.grad(g)
        if pc.kind == "conv":
            table.add(finish, batched.FINISH_ROW, pc.cout, pc.cin * pc.taps * 4, self.dwp, g, v, dv, dg,
                      ints=(0, pc.cout, pc.cin, pc.taps, self.rows, pc.cin_p, pc.cout, 1, 0, 0, 0, 0, 1),
                      tab=range(pc.taps))
        else:
            k = m.kernel_size[0]
            nshift, smin = c_int(), c_int()
            _lib.check(_lib.lib().hg_convtr1d_geometry(k, pc.stride, m.padding[0], byref(nshift), byref(smin)))
            table.add(finish, batched.FINISH_ROW, pc.cin, pc.cout * k * 4, self.dwp, g, v, dv, dg,
                      ints=(1, pc.cin, pc.cout, k, pc.stride * pc.cout_p, pc.cin_p, 0, 1, pc.stride, m.padding[0],
                            smin.value, pc.cout_p, 1))

    def wgrad(self, L, x, dy, batch: int, t: int) -> None:
        """x bf16 [B][t][cin_p] (the forward input), dy bf16 [B][t][rows] -> dwp (+=)"""
        pc = self.pc
        _lib.check(L.hg_conv1d_wgrad(_p(x), _p(dy), batch, t, pc.cin_p, t, t, 1, self.rows, pc.taps, 1, pc.dil,
                                     pc.pad_left, self.dwp.data_ptr(), 1, _stream()), "hg_conv1d_wgrad")

    def bias_dst(self, c: int) -> int:
        """pointer of bias.grad when the producer of this layer's output gradient can add its fp32 column sums
        straight into it (no channel padding: c output columns == cout), else 0 -> bias_grad() runs afterwards"""
        b = self.pc.module.bias
        return self.flat.grad(b).data_ptr() if (b is not None and c == self.pc.cout) else 0

    def bias_grad(self, L, dy, batch: int, t: int, c: int) -> None:
        """bias.grad (+)= column sums of dy [B][t][c] — only for layers with channel padding (V2's 16-channel stage);
        every other bias gradient comes from the fp32 accumulators of the launch that produced dy (bias_dst)"""
        b = self.pc.module.bias
        if b is None or self.bias_dst(c):
            return
        if c == self.pc.cout:
            _lib.check(L.hg_colsum_bf16(_p(dy), batch, t, t, c, 1, self.flat.grad(b).data_ptr(), _stream()),
                       "hg_colsum_bf16")
        else:
            if self.db is None:
                self.db = torch.zeros(c, dtype=torch.float32, device=dy.device)
            _lib.check(L.hg_colsum_bf16(_p(dy), batch, t, t, c, 0, self.db.data_ptr(), _stream()), "hg_colsum_bf16")
            self.flat.grad(b).add_(self.db[: self.pc.cout])

    def dgrad(self, L, dy, batch: int, t: int, out, mask=None, slope: float = LRELU_SLOPE, res0=None, res1=None,
              res2=None, scale: float = 1.0, bias_dsts=()) -> None:
        """bias_dsts: up to three bias.grad pointers (bias_dst) of the layer(s) whose output gradient `out` is"""
        pc = self.pc
        bd = [d for d in bias_dsts if d] + [0, 0, 0]
        _lib.check(L.hg_conv1d_dgrad(_p(dy), self.wd.data_ptr(), batch, t, t, self.rows, t, t, 1, 0, pc.cin_p,
                                     pc.taps, pc.dil, self.dgrad_pad, _p(mask), slope, 0, 0, 0.0, _p(res0), _p(res1),
                                     _p(res2), scale, _p(out), 0, 0, 1, 0, 0, bd[0], bd[1], bd[2], 0, _stream()),
                   "hg_conv1d_dgrad")

    def to_param_grads(self, L) -> None:
        """packed dW -> (weight_g.grad, weight_v.grad) or weight.grad, one fused launch (hg_wgrad_finish_*)"""
        pc = self.pc
        m = pc.module
        g, v = _g_v(m)
        gp, dgp = (0, 0) if g is None else (g.data_ptr(), self.flat.grad(g).data_ptr())
        dvp = self.flat.grad(v).data_ptr()
        if pc.kind == "conv":
            _lib.check(L.hg_wgrad_finish_conv(self.dwp.data_ptr(), pc.cout, pc.cin, pc.taps, self.rows, pc.cin_p,
                                              pc.cout, 1, None, v.data_ptr(), gp, 1, dvp, dgp,
                                              _stream()), "hg_wgrad_finish_conv")
        else:
            _lib.check(L.hg_wgrad_finish_convtr(self.dwp.data_ptr(), pc.cin, pc.cout, m.kernel_size[0], pc.stride,
                                                m.padding[0], pc.cin_p, pc.cout_p, v.data_ptr(), gp, 1,
                                                dvp, dgp, _stream()), "hg_wgrad_finish_convtr")


def _route_weight_grad(L, flat: FlatParams, m: nn.Module, dw: torch.Tensor, d0: int, rest: int,
                       accumulate: bool = False) -> None:
    """dw fp32 (dense, parameter layout, first d0*rest elements of `dw`) -> the module's parameter gradients in
    `flat`'s gradient buffer."""
    g, v = _g_v(m)
    if g is not None:
        _lib.check(L.hg_weight_norm_bwd(dw.data_ptr(), v.data_ptr(), g.data_ptr(), d0, rest, 1 if accumulate else 0,
                                        flat.grad(v).data_ptr(), flat.grad(g).data_ptr(), _stream()),
                   "hg_weight_norm_bwd")
    else:
        src = dw[: d0 * rest].view(v.shape)
        if accumulate:
            flat.grad(v).add_(src)
        else:
            flat.grad(v).copy_(src)


class GeneratorTrainer:
    """Training-mode forward (every conv input kept in HBM) and hand-written backward of one Generator."""

    def __init__(self, gen: Generator, device, bind: bool = True):
        """bind=False: the autograd path — gradients go to a private flat buffer, parameters stay torch's, and the
        gradient at the input mel can be produced (conv_pre gets a data-gradient bank)."""
        self.gen, self.device = gen, device
        self.flat = FlatParams(gen, device, bind)
        gen._drop_engines()
        self.eng = gen._engine(device)
        e = self.eng
        self.g_pre = _GenLayerGrad(e.pre, device, self.flat, need_dgrad=not bind)
        self.g_ups = [_GenLayerGrad(pc, device, self.flat) for pc in e.ups]
        self.g_blocks = [[_GenLayerGrad(pc, device, self.flat) for pc in blk] for blk in e.blocks]
        layers = [self.g_pre] + self.g_ups + [x for b in self.g_blocks for x in b]
        self.dwp_flat = torch.zeros(sum(gl.dwp_numel for gl in layers), dtype=torch.float32, device=device)
        off = 0
        for gl in layers:
            gl.dwp = self.dwp_flat[off:off + gl.dwp_numel]
            off += gl.dwp_numel
        # the data-gradient banks of every layer / the finish of every packed weight gradient: one launch each
        from . import batched
        # (finishes go per MRF branch / upsampling conv, launched on the weight-gradient lanes as soon as that
        # branch's wgrads are queued: only the first stage's are left when the data-gradient chain ends)
        self.table = batched.JobTable(device)
        self.g_pre.add_jobs(self.table, "finish_pre")
        for i, gl in enumerate(self.g_ups):
            gl.add_jobs(self.table, f"finish_up{i}")
        nk_ = gen.num_kernels
        for n, blk in enumerate(self.g_blocks):
            for gl in blk:
                gl.add_jobs(self.table, f"finish_{n // nk_}_{n % nk_}")
        self.table.finalize()
        # stream lanes: 0 .. nk-2 = MRF branches beside the main stream, W_LANE + j = weight-gradient work of branch j
        nk = gen.num_kernels
        self.W_LANE = max(1, nk - 1)
        self.lanes = _Lanes(self.W_LANE + nk, device, [-1] * self.W_LANE + [0] * nk)
        post = gen.conv_post
        self.post_dw = torch.zeros(e.post_cin_p, post.kernel_size[0], dtype=torch.float32, device=device)
        self.post_db = torch.zeros(1, dtype=torch.float32, device=device)
        self.ws: Dict[Tuple[int, int], dict] = {}
        self.two_conv = isinstance(gen.resblocks[0], ResBlock1)
        if gen.num_kernels > 3:
            raise NotImplementedError("training path supports up to 3 MRF branches (V1/V2/V3)")

    def invalidate(self) -> None:
        """parameters were updated in place through raw pointers (AdamW kernel): force a re-pack"""
        engines = [self.eng] + [e for e in self.gen.__dict__.get("_hg_engines", {}).values() if e is not self.eng]
        for e in engines:      # the module API (`generator(x)` in eval / validation) may hold engines of its own
            e.invalidate()

    def _workspace(self, b: int, frames: int) -> dict:
        ws = self.ws.get((b, frames))
        if ws is not None:
            return ws
        e, gen, dev = self.eng, self.gen, self.device
        bf = lambda *shape: torch.empty(*shape, dtype=torch.bfloat16, device=dev)
        nk = gen.num_kernels
        ws = {"mel": bf(b, frames, e.pre.cin_p), "pre_act": bf(b, frames, e.pre.cout_p), "stages": []}
        t = frames
        for i, up in enumerate(e.ups):
            t_in = t
            t *= up.stride
            c = up.cout_p
            steps = len(e.blocks[i * nk]) // (2 if self.two_conv else 1)
            mk = lambda: bf(b, t, c)
            # The MRF branches run on parallel stream lanes and the weight-gradient launches beside the data-gradient
            # chain, so nothing is ping-ponged: every branch / step owns its buffers.
            st = {"t_in": t_in, "t": t, "c": c, "steps": steps, "x_raw": mk(), "xa0": mk(), "stage_act": mk(),
                  "raw": [[mk(), mk()] for _ in range(nk)], "r": [mk() for _ in range(max(1, nk - 1))],
                  # saved conv inputs: xa[j][s] for s >= 1 (s = 0 is the shared xa0), t1[j][s]
                  "xa": [[None] + [mk() for _ in range(steps - 1)] for _ in range(nk)],
                  "t1": [[mk() for _ in range(steps)] for _ in range(nk)] if self.two_conv else None,
                  # gradients: g0 at the stage output, gs[j][s] at the input of step s of branch j, gt1[j][s]
                  "g0": mk(), "gs": [[mk() for _ in range(steps)] for _ in range(nk)],
                  "gt1": [[mk() for _ in range(steps)] for _ in range(nk)] if self.two_conv else None}
            ws["stages"].append(st)
        ws["y"] = torch.empty(b, 1, t, dtype=torch.float32, device=dev)
        ws["dpre"] = torch.empty(b, t, dtype=torch.float32, device=dev)
        ws["g_pre"] = bf(b, frames, e.pre.cout_p)
        ws["t_out"] = t
        if len(self.ws) >= 4:
            self.ws.pop(next(iter(self.ws)))
        self.ws[(b, frames)] = ws
        return ws

    # ---- forward -------------------------------------------------------------------------------------------
    def _branch_forward(self, L, st, j: int, packs, b: int, t: int, stop_before_last: bool):
        """steps of MRF branch j; returns the (src, conv, residual) of its final launch when stop_before_last"""
        cur_raw, cur_act = st["x_raw"], st["xa0"]
        for s in range(st["steps"]):
            last = s == st["steps"] - 1
            if self.two_conv:
                _conv(L, cur_act, packs[2 * s], b, t, out_act=st["t1"][j][s])
                src, pc = st["t1"][j][s], packs[2 * s + 1]
            else:
                src, pc = cur_act, packs[s]
            if not last:
                nr, na = st["raw"][j][s & 1], st["xa"][j][s + 1]
                _conv(L, src, pc, b, t, res=(cur_raw, None, None), out_raw=nr, out_act=na)
                cur_raw, cur_act = nr, na
            elif stop_before_last:
                return src, pc, cur_raw
            else:
                _conv(L, src, pc, b, t, res=(cur_raw, None, None), out_raw=st["r"][j])
        return None

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """mel fp32 [B,80,F] -> waveform fp32 [B,1,T] (engine-owned buffer), keeping what backward needs."""
        L = _lib.lib()
        e, gen = self.eng, self.gen
        lanes = self.lanes
        b, c, frames = x.shape
        xin = x.contiguous().float()
        ws = self._workspace(b, frames)
        self.cur = ws
        main = torch.cuda.current_stream()
        lanes.fork()
        # after an optimizer update every filter bank is re-folded and re-packed: ONE launch over the engine's job table
        e.refresh()
        _lib.check(L.hg_ncl_to_nlc(xin.data_ptr(), b, c, frames, e.pre.cin_p, ws["mel"].data_ptr(), 0, 0.0, _stream()),
                   "hg_ncl_to_nlc")
        _conv(L, ws["mel"], e.pre, b, frames, out_act=ws["pre_act"])
        lanes.join()
        lanes.streams[self.W_LANE].wait_stream(main)
        with lanes.lane(self.W_LANE):            # the data-gradient filter banks are not needed before backward
            self.table.launch("dgrad")
        cur, t = ws["pre_act"], frames
        nk = gen.num_kernels
        for i, up in enumerate(e.ups):
            st = ws["stages"][i]
            _conv(L, cur, up, b, t, out_raw=st["x_raw"], out_act=st["xa0"])
            t = st["t"]
            out_slope = 0.01 if i == len(e.ups) - 1 else LRELU_SLOPE
            for j in range(nk - 1):              # branches 0 .. nk-2 on their own lanes
                lanes.streams[j].wait_stream(main)
                with lanes.lane(j):
                    self._branch_forward(L, st, j, e.blocks[i * nk + j], b, t, False)
            src, pc, cur_raw = self._branch_forward(L, st, nk - 1, e.blocks[i * nk + nk - 1], b, t, True)
            for j in range(nk - 1):
                main.wait_stream(lanes.streams[j])
            others = tuple(st["r"][q] for q in range(nk - 1)) + (None,) * (3 - nk)
            _conv(L, src, pc, b, t, res=(cur_raw,) + others[:2], scale=1.0 / nk, out_act=st["stage_act"],
                  slope=out_slope)
            cur = st["stage_act"]
        post = gen.conv_post
        _lib.check(L.hg_conv_post_tanh_fwd(cur.data_ptr(), e.post_w.data_ptr(), e.post_b.data_ptr(), b, t,
                                           e.post_cin_p, post.kernel_size[0], ws["y"].data_ptr(), _stream()),
                   "hg_conv_post_tanh_fwd")
        lanes.join()
        return ws["y"]

    # ---- backward ------------------------------------------------------------------------------------------
    def _side(self, L, lane: int, producer, fn) -> None:
        """run fn() (weight / bias gradient work) on a side lane once `producer` (a stream) reached this point"""
        s = self.lanes.streams[lane]
        s.wait_stream(producer)
        with torch.cuda.stream(s):
            fn()

    def _branch_backward(self, L, st, i: int, j: int, b: int, t: int, c: int, g0, extra, up_bias: int = 0):
        """data-gradient chain of MRF branch j on the current stream; its weight / bias gradients on lane W_LANE + j.
        `extra` = gradients of the other branches to add into the last launch (None: write gs[j][0] alone).
        Every data-gradient launch also sums its fp32 output columns into the bias gradient of the conv that
        produced the tensor it differentiates (up_bias: the upsampling conv's, for the branch-summing last launch)."""
        gl = self.g_blocks[i * self.gen.num_kernels + j]
        wl = self.W_LANE + j
        g = g0
        here = torch.cuda.current_stream()
        for s in reversed(range(st["steps"])):
            xa = st["xa0"] if s == 0 else st["xa"][j][s]
            out = st["gs"][j][s]
            r1, r2 = (extra if (s == 0 and extra is not None) else (None, None))
            # `out` is the gradient at the output of the previous step's last conv (s > 0) or of the upsampling conv
            prev = (gl[2 * s - 1] if self.two_conv else gl[s - 1]) if s > 0 else None
            out_bias = (prev.bias_dst(c),) if prev is not None else ((up_bias,) if extra is not None else ())
            if self.two_conv:
                c1, c2 = gl[2 * s], gl[2 * s + 1]
                t1, gt1 = st["t1"][j][s], st["gt1"][j][s]

                def w2(c2=c2, t1=t1, g=g):
                    c2.bias_grad(L, g, b, t, c)
                    c2.wgrad(L, t1, g, b, t)
                self._side(L, wl, here, w2)
                c2.dgrad(L, g, b, t, gt1, mask=t1, bias_dsts=(c1.bias_dst(c),))

                def w1(c1=c1, xa=xa, gt1=gt1):
                    c1.bias_grad(L, gt1, b, t, c)
                    c1.wgrad(L, xa, gt1, b, t)
                self._side(L, wl, here, w1)
                c1.dgrad(L, gt1, b, t, out, mask=xa, res0=g, res1=r1, res2=r2, bias_dsts=out_bias)
            else:
                cc = gl[s]

                def w0(cc=cc, xa=xa, g=g):
                    cc.bias_grad(L, g, b, t, c)
                    cc.wgrad(L, xa, g, b, t)
                self._side(L, wl, here, w0)
                cc.dgrad(L, g, b, t, out, mask=xa, res0=g, res1=r1, res2=r2, bias_dsts=out_bias)
            g = out
        # this branch's packed weight gradients are all queued on its lane: finish them there
        self._side(L, wl, here, lambda: self.table.launch(f"finish_{i}_{j}"))
        return g

    def _last_conv_bias_dsts(self, i: int, c: int):
        """bias.grad pointers of the last conv of every MRF branch of stage i (they share one output gradient, g0)"""
        nk = self.gen.num_kernels
        d = [self.g_blocks[i * nk + j][-1].bias_dst(c) for j in range(nk)]
        return (d + [0, 0, 0])[:3]

    def backward(self, dy: torch.Tensor, dx_mel: Optional[torch.Tensor] = None) -> None:
        """dy fp32 [B,T] (or [B,1,T]): gradient at the waveform of the LAST forward -> every parameter's gradient
        buffer.  dx_mel (optional, fp32 [B, cin_p, F], autograd path): receives the gradient at the input mel."""
        L = _lib.lib()
        e, gen, ws = self.eng, self.gen, self.cur
        lanes = self.lanes
        b, frames = ws["mel"].shape[0], ws["mel"].shape[1]
        nk = gen.num_kernels
        dy = dy.reshape(b, -1).contiguous().float()
        t = ws["t_out"]
        post = gen.conv_post
        stages = ws["stages"]
        last = stages[-1]
        main = torch.cuda.current_stream()
        self.post_dw.zero_()
        self.post_db.zero_()
        self.dwp_flat.zero_()          # every wgrad / finish / bias kernel below accumulates
        self.flat.g.zero_()
        lanes.fork()
        # conv_post + tanh; the kernel also applies the slope-0.01 leaky_relu mask of the last stage, the 1 / nk of
        # the MRF mean (earlier stages get it from the ups dgrad scale) and sums the bias gradients of the branches'
        # last convs (they all see this gradient) from its fp32 values
        bd = self._last_conv_bias_dsts(len(e.ups) - 1, last["c"])
        _lib.check(L.hg_conv_post_tanh_bwd(last["stage_act"].data_ptr(), e.post_w.data_ptr(), ws["y"].data_ptr(),
                                           dy.data_ptr(), b, t, e.post_cin_p, post.kernel_size[0], 0.01, 1.0 / nk,
                                           last["g0"].data_ptr(), ws["dpre"].data_ptr(), self.post_dw.data_ptr(),
                                           self.post_db.data_ptr(), bd[0], bd[1], bd[2], _stream()),
                   "hg_conv_post_tanh_bwd")

        def post_grads():
            cin, k = post.in_channels, post.kernel_size[0]
            _route_weight_grad(L, self.flat, post, self.post_dw[:cin].contiguous(), 1, cin * k)
            self.flat.grad(post.bias).copy_(self.post_db)      # flat.g was zeroed: plain stores here
        self._side(L, self.W_LANE, main, post_grads)
        for i in reversed(range(len(e.ups))):
            st = stages[i]
            t, c = st["t"], st["c"]
            g0 = st["g0"]
            # branches 0 .. nk-2 on their own lanes, the last one here; it adds the others into its final launch
            for j in range(nk - 1):
                lanes.streams[j].wait_stream(main)
                with lanes.lane(j):
                    self._branch_backward(L, st, i, j, b, t, c, g0, None)
            # the last branch's chain up to (not including) its final launch must not wait for the others: run it,
            # then join right before the final launch.  _branch_backward issues the final launch itself, so the join
            # happens first — the other branches are the same length, little is lost.
            for j in range(nk - 1):
                main.wait_stream(lanes.streams[j])
            others = [st["gs"][j][0] for j in range(nk - 1)] + [None, None]
            up = self.g_ups[i]
            dx_raw = self._branch_backward(L, st, i, nk - 1, b, t, c, g0, (others[0], others[1]), up.bias_dst(c))
            t_in = st["t_in"]
            up_in = ws["pre_act"] if i == 0 else stages[i - 1]["stage_act"]

            def up_grads(up=up, dx_raw=dx_raw, up_in=up_in, t=t, c=c, t_in=t_in):
                up.bias_grad(L, dx_raw, b, t, c)               # dx_raw as [B][t][c]: phases fold into the rows
                up.wgrad(L, up_in, dx_raw, b, t_in)            # dy viewed as [B][t_in][stride * c]
                self.table.launch(f"finish_up{i}")
            self._side(L, self.W_LANE, main, up_grads)
            if i > 0:
                up.dgrad(L, dx_raw, b, t_in, stages[i - 1]["g0"], mask=up_in, scale=1.0 / nk,
                         bias_dsts=self._last_conv_bias_dsts(i - 1, stages[i - 1]["c"]))
            else:
                up.dgrad(L, dx_raw, b, t_in, ws["g_pre"], mask=up_in, bias_dsts=(self.g_pre.bias_dst(e.pre.cout_p),))
                self.g_pre.bias_grad(L, ws["g_pre"], b, frames, e.pre.cout_p)
                self.g_pre.wgrad(L, ws["mel"], ws["g_pre"], b, frames)
                if dx_mel is not None:
                    gm = ws.get("g_mel")
                    if gm is None:
                        gm = ws["g_mel"] = torch.empty_like(ws["mel"])
                    self.g_pre.dgrad(L, ws["g_pre"], b, frames, gm)
                    _lib.check(L.hg_nlc_to_ncl(gm.data_ptr(), b, frames, e.pre.cin_p, dx_mel.data_ptr(), _stream()),
                               "hg_nlc_to_ncl")
                self.table.launch("finish_pre")
        lanes.join()


# ------------------------------------------------------------------------------------------------ discriminators
class _DiscBwdLayer:
    """Data-gradient side of one wide discriminator conv: the polyphase / flipped filter bank and its launch."""

    def __init__(self, layer: _DiscLayer, device):
        self.layer = layer
        s, k, pad = layer.stride, layer.k, layer.pad
        L = _lib.lib()
        nshift, smin = c_int(), c_int()
        _lib.check(L.hg_convtr1d_geometry(k, s, pad, byref(nshift), byref(smin)))
        self.nshift, self.smin = nshift.value, smin.value
        self.pad_left = -self.smin
        self.grouped = layer.groups > 1
        self.cout_tile = (layer.cout // layer.groups) * layer.merge
        self.w = torch.empty(self.nshift, s * layer.cin, self.cout_tile, dtype=torch.bfloat16, device=device)

    def pack(self, w_eff: torch.Tensor, w_fwd_packed=None) -> None:
        """w_eff fp32 [cout][cin/groups][k] (effective weight) -> the data-gradient filter bank (hg_pack_disc_weight).
        w_fwd_packed is not read: the bank is derived from w_eff alone."""
        layer = self.layer
        _lib.check(_lib.lib().hg_pack_disc_weight(w_eff.data_ptr(), layer.cout, layer.cin, layer.groups, layer.merge,
                                                  layer.k, layer.stride, layer.pad, 0, self.w.data_ptr(), _stream()),
                   "hg_pack_disc_weight")

    def dgrad(self, L, dy, nseq: int, t_dy_valid: int, t_dy_rows: int, rows_in: int, act_g, act_r, fm_coef: float,
              out, st, flat_h_in: Optional[int] = None, bias_dst: int = 0, pre_add=None) -> None:
        """out[nseq][rows_in][cin] = (conv^T(dy) + fm_coef * sgn(act_g - act_r) + pre_add) * lrelu'(act_g).
        flat_h_in given: the nseq sequences are laid end to end (pitch t_dy_rows output rows / rows_in input rows
        each, zero gap rows) and run as ONE long sequence; only positions < flat_h_in of each are stored.
        bias_dst: fp32 [cin] bias gradient of the layer that produced act_g, += column sums of `out` (fp32)."""
        layer = self.layer
        s = layer.stride
        vrows = rows_in // s
        batch, t_valid, t_rows, t_out, seq = nseq, t_dy_valid, t_dy_rows, vrows, (0, 0, 1, 0)
        if flat_h_in is not None:
            batch, t_valid, t_rows, t_out = 1, nseq * t_dy_rows, nseq * t_dy_rows, nseq * vrows
            seq = (vrows, flat_h_in, s, layer.cin)
        _lib.check(L.hg_conv1d_dgrad(_p(dy), self.w.data_ptr(), batch, t_valid, t_rows, layer.cout, t_out, t_out,
                                     layer.groups_eff if self.grouped else 1,
                                     layer.cin_tile if self.grouped else 0, s * layer.cin, self.nshift, 1,
                                     self.pad_left, _p(act_g), LRELU_SLOPE, _p(act_r),
                                     _p(act_g) if act_r is not None else 0, fm_coef, 0, 0, 0, 1.0, _p(out), *seq,
                                     _p(pre_add), bias_dst, 0, 0, layer.cin, st),
                   "hg_conv1d_dgrad")


class _SubDiscTrainer:
    """One DiscriminatorP / DiscriminatorS: batched (real ++ generated) forward with saved activations, losses on
    the internal layout, and the hand-written backward."""

    W_CHAINS = 4

    def __init__(self, disc: nn.Module, device, flat: FlatParams, boost: int = 0):
        """flat: the FlatParams whose gradient buffer receives this sub-discriminator's parameter gradients.
        boost: added to the CUDA stream priorities of every lane of this sub-discriminator (negative = more urgent):
        the sub-discriminator with the longest chain (the spectral-norm scale) is the step's critical path, so its
        kernels — its weight-gradient lane included — are placed ahead of the other sub-discriminators'."""
        self.disc, self.device, self.flat = disc, device, flat
        self.period = getattr(disc, "period", 1)
        convs = list(disc.convs)
        self.mods = convs + [disc.conv_post]
        m0 = convs[0]
        self.first = (m0.kernel_size[0], m0.stride[0], m0.padding[0], m0.out_channels)
        groups = lambda m: getattr(m, "groups", 1)
        self.mids = [_DiscLayer(m.in_channels, m.out_channels, m.kernel_size[0], m.stride[0], m.padding[0], groups(m))
                     for m in convs[1:]]
        self.bwd = [_DiscBwdLayer(l, device) for l in self.mids]
        self.kpost = disc.conv_post.kernel_size[0]
        self.spectral = hasattr(m0, "weight_orig")
        # the spectral-norm scale runs its real / generated halves as two parts with their own sigma (and their own
        # data-gradient filter banks), on two lanes; lane 0 is the parameter-gradient lane of this sub-discriminator
        self.bwd_parts = [self.bwd] + ([[_DiscBwdLayer(l, device) for l in self.mids]] if self.spectral else [])
        self.lanes = _Lanes(2, device, [0 + boost, -1 + boost])   # 0: parameter-gradient lane, 1: second data-gradient chain
        n_prep = 8 if self.spectral else 4                        # spectral norm: one power-iteration chain per layer
        self.prep = _Lanes(n_prep, device, [-1 + boost] * n_prep)  # weight preparation / data-gradient packs
        self._prefetched = None
        # spectral norm: every layer's parameter-gradient chain (wgrad -> unpack -> <dw,w> -> apply, for both halves)
        # is independent of the other layers': spread over W_CHAINS lanes instead of one.  (One lane made this the
        # longest dependent chain of the whole step: 3.9 ms for 2 x 8 layers, profiles/r02_summary.md section 2.)
        # weight_norm sub-discriminators: one lane (measured with 1 / 2 / 4 / 8: 12.01 / 12.01 / 12.06-12.12 / 12.10 ms —
        # their chains are short and the phase is bound by SM-time)
        self.n_chains = self.W_CHAINS if self.spectral else 1
        self.wl = _Lanes(self.n_chains, device, [0 + boost] * self.n_chains)
        self._scr = {}
        self.ws = {}
        # packed fp32 weight gradients, one region per wide layer (zeroed once per backward; the wgrad launches
        # accumulate)
        sizes = [l.k * l.cout * l.cin_tile for l in self.mids]
        self.dwp_flat = torch.zeros(sum(sizes), dtype=torch.float32, device=device)
        self.dwps, off = [], 0
        for n in sizes:
            self.dwps.append(self.dwp_flat[off:off + n])
            off += n
        self._tables = {}
        self.db = torch.zeros(1024, dtype=torch.float32, device=device)
        self.db_unused = torch.zeros(1024, dtype=torch.float32, device=device)    # the first conv's discarded bias column
        self.wbufs = {}
        self.fwd_valid = self.dgrad_valid = False
        self.W_cached = None

    def invalidate(self) -> None:
        """the parameters changed (optimizer update / load_state_dict): re-fold and re-pack on next use"""
        self.fwd_valid = self.dgrad_valid = False

    # ---- weights -------------------------------------------------------------------------------------------
    def _scratch_of(self, chain: int) -> torch.Tensor:
        """fp32 scratch of parameter-gradient chain `chain` (0: conv_post, 1..nl: the wide layers from the last to the
        first, nl + 1: the first conv), sized for that layer's weight: the chains run side by side"""
        buf = self._scr.get(chain)
        if buf is None:
            nl = len(self.mids)
            m = self.mods[-1] if chain == 0 else self.mods[0] if chain == nl + 1 else self.mods[1 + nl - chain]
            w = m.weight_orig if hasattr(m, "weight_orig") else m.weight_v if hasattr(m, "weight_v") else m.weight
            buf = self._scr[chain] = torch.empty(w.numel(), dtype=torch.float32, device=self.device)
        return buf

    def _weights(self, part: int):
        """per-part persistent buffers of every layer's effective fp32 weight and forward GEMM pack; _weights_layer
        and the table's "fwd" launch fill them"""
        bufs = self.wbufs.get(part)
        if bufs is None:
            bufs = {"eff": [], "fwd": []}
            for li, m in enumerate(self.mods):
                _, v = _g_v(m) if not hasattr(m, "weight_orig") else (None, m.weight_orig)
                bufs["eff"].append(torch.empty(v.shape[0], v.shape[1], v.shape[2] if v.dim() > 2 else 1,
                                               dtype=torch.float32, device=self.device))
                if 1 <= li <= len(self.mids):
                    layer = self.mids[li - 1]
                    bufs["fwd"].append(torch.empty(layer.k, layer.cout, layer.cin_tile, dtype=torch.bfloat16,
                                                   device=self.device))
                else:
                    bufs["fwd"].append(None)
            self.wbufs[part] = bufs
        return {"eff": bufs["eff"], "fwd": bufs["fwd"], "sn": [None] * len(self.mods)}

    def _table(self, part: int):
        """Job table of part / call slot `part` (batched.py): phase "fwd" = weight_norm fold -> effective fp32 weight +
        forward bank of every layer (spectral-norm layers: forward bank from the effective weight their power
        iteration produced), "dgrad" = the polyphase data-gradient banks.  One launch each instead of one per layer."""
        t = self._tables.get(part)
        if t is not None:
            return t
        from . import batched
        L = _lib.lib()
        bufs = self.wbufs[part]
        t = batched.JobTable(self.device)
        nl = len(self.mids)
        self.untiled = []                         # layers whose data-gradient bank does not tile: packed per layer
        for li, m in enumerate(self.mods):
            layer = self.mids[li - 1] if 1 <= li <= nl else None
            sn = hasattr(m, "weight_orig")
            if sn and layer is None:
                continue                          # first / last conv of the spectral-norm scale: eff is all they need
            g, v = (None, bufs["eff"][li]) if sn else _g_v(m)
            cout = v.shape[0]
            cin_g, k = (layer.cin // layer.groups, layer.k) if layer is not None else (v.shape[1], v.numel() // (v.shape[0] * v.shape[1]))
            ints = (cout, cin_g, k, layer.merge if layer else 1, (layer.cout // layer.groups) if layer else cout,
                    layer.cin_tile if layer else cin_g)
            t.add("fwd", batched.DISC_ROW, cout, cin_g * k * 4 if layer is not None else 0, v, g,
                  dst0=None if sn else bufs["eff"][li], dst1=bufs["fwd"][li] if layer is not None else None,
                  ints=ints, tab=layer.order if layer is not None else ())
            if layer is None:
                continue
            bl = self._bwd_bank(part)[li - 1]
            cout_tile = (layer.cout // layer.groups) * layer.merge
            tci = 32 if layer.k <= 10 else 8
            while tci > 2 and (cin_g % tci or layer.cin % tci):
                tci >>= 1
            smem = 32 * (tci * layer.k + 1) * 4
            if cin_g % tci == 0 and layer.cin % tci == 0 and cout_tile % 32 == 0 and smem <= 48 * 1024:
                t.add("dgrad", batched.DISC_DGRAD_TILE, (layer.cin // tci) * (cout_tile // 32), smem, bufs["eff"][li],
                      dst0=bl.w, ints=(layer.cout, cin_g, layer.k, layer.merge, layer.cout // layer.groups, layer.cin,
                                       layer.stride, layer.pad, bl.nshift, bl.smin, cout_tile, tci, layer.cin // tci))
            else:
                self.untiled.append(li - 1)
        self._tables[part] = t.finalize()
        return t

    def _prepare_weights(self, part: int) -> dict:
        """effective weights + forward banks of part `part` on the current stream: spectral-norm layers run their
        power iteration (one per call in train mode, like the reference's hook), then ONE batched launch folds /
        packs every layer"""
        W = self._weights(part)
        if self.spectral:
            for li in range(len(self.mods)):
                self._weights_layer(W, self.wbufs[part], li)
        self._table(part).launch("fwd")
        return W

    def prefetch_weights(self) -> None:
        """Spectral norm only: queue the NEXT forward's power iterations (both halves) and forward banks on the prep
        lanes, forked from the current stream, without joining them back — forward() waits for them.  The training
        step calls this before the generator's forward: the discriminator-step weights depend on nothing the
        generator produces, and inside the discriminator phase these small launches wait for SMs behind the other
        lanes' persistent tensor-core kernels (measured: 0.98 -> 3.0 ms for chains that take 0.2 ms on a quiet GPU)."""
        if not self.spectral:
            return
        Ws = [self._weights(pi) for pi in range(2)]
        self.prep.fork()
        for li in range(len(self.mods)):
            with self.prep.lane(li):
                for pi, W in enumerate(Ws):
                    self._weights_layer(W, self.wbufs[pi], li)
        p0 = self.prep.streams[0]
        for s_ in self.prep.streams[1:]:
            p0.wait_stream(s_)
        with torch.cuda.stream(p0):
            for pi in range(2):
                self._table(pi).launch("fwd")
        self._prefetched = Ws

    def _weights_layer(self, ws, bufs, li: int) -> None:
        """fold (weight norm) or power-iterate (spectral norm) layer li into its effective fp32 weight"""
        L = _lib.lib()
        st = _stream()
        m = self.mods[li]
        eff = bufs["eff"][li]
        if hasattr(m, "weight_orig"):
            wo = m.weight_orig
            rows, cols = wo.shape[0], wo.numel() // wo.shape[0]
            snb = bufs.setdefault("sn", {}).get(li)
            if snb is None:
                f32 = lambda n: torch.empty(n, dtype=torch.float32, device=self.device)
                snb = (f32(rows), f32(cols), f32(1), f32(rows + cols + 4))     # u, v, sigma of this call; workspace
                bufs["sn"][li] = snb
            # one power iteration per call in train mode, u / v buffers updated in place (hg_spectral_norm_fwd);
            # the copies are what the backward of THIS call's weights needs (the next call moves u, v on)
            _lib.check(L.hg_spectral_norm_fwd(wo.data_ptr(), m.weight_u.data_ptr(), m.weight_v.data_ptr(), rows,
                                              cols, 1 if m.training else 0, eff.data_ptr(), snb[2].data_ptr(),
                                              snb[0].data_ptr(), snb[1].data_ptr(), snb[3].data_ptr(), st),
                       "hg_spectral_norm_fwd")
            ws["sn"][li] = snb
        else:
            g, v = _g_v(m)
            _lib.check(L.hg_fold_weight_norm(v.data_ptr(), 0 if g is None else g.data_ptr(), v.shape[0],
                                             v.numel() // v.shape[0], eff.data_ptr(), st), "hg_fold_weight_norm")

    def _geometry(self, nb: int, t: int, slot: int = 0):
        key = (nb, t, slot)
        g = self.ws.get(key)
        if g is not None:
            return g
        dev, period = self.device, self.period
        k0, s0, p0, c0 = self.first
        h = (t + period - 1) // period
        if h * period - t >= t:
            raise RuntimeError("reflect padding needs n_pad < t (reference F.pad behaviour)")
        hh = (h + 2 * p0 - k0) // s0 + 1
        hs, cs = [hh], [c0]
        for layer in self.mids:
            hh = (hh + 2 * layer.pad - layer.k) // layer.stride + 1
            hs.append(hh)
            cs.append(layer.cout)
        geo = [(h_, p_, c_) for h_, p_, c_ in zip(hs, self._flat_pitches(hs), cs)]
        nseq = nb * period
        g = {"geo": geo, "nseq": nseq,
             "act": [torch.zeros(nseq, r, c, dtype=torch.bfloat16, device=dev) for _, r, c in geo],
             "grad": [torch.zeros(nseq, r, c, dtype=torch.bfloat16, device=dev) for _, r, c in geo],
             "logit": torch.empty(nseq, geo[-1][0], dtype=torch.float32, device=dev),
             "dlogit": torch.empty(nseq, geo[-1][0], dtype=torch.float32, device=dev)}
        if len(self.ws) >= 8:
            self.ws.pop(next(iter(self.ws)))
        self.ws[key] = g
        return g

    def _flat_pitches(self, hs: List[int]) -> List[int]:
        """Rows per sequence of every activation buffer when the sequences of a layer are laid end to end and run as
        ONE long sequence (the late layers have 10..51 rows per sequence; 128-row tiles would be mostly empty
        otherwise).  Buffer l feeds layer l (stride s_l) whose output is buffer l+1, so pitch_l = s_l * pitch_{l+1};
        the zero rows between two sequences must cover the padding every conv / data-gradient tap reaches into."""
        def chain(p_last):
            ps = [p_last]
            for layer in reversed(self.mids):
                ps.insert(0, ps[0] * layer.stride)
            return ps

        def ok(ps):
            for li, (layer, bl) in enumerate(zip(self.mids, self.bwd)):
                h_in, p_in, h_out, p_out, s = hs[li], ps[li], hs[li + 1], ps[li + 1], layer.stride
                if p_in - h_in < layer.pad:                                   # left padding of the next sequence
                    return False
                if (h_out - 1) * s + layer.k - 1 - layer.pad > p_in - 1:        # right reach of the last output
                    return False
                smax = bl.smin + bl.nshift - 1
                if p_out - h_out < -bl.smin:                                   # data gradient: taps before row 0
                    return False
                if (h_in + s - 1) // s - 1 + smax > p_out - 1:                  # ... and past the last row
                    return False
            return True

        p_last = hs[-1] + 1
        while not ok(chain(p_last)):
            p_last += 1
        return chain(p_last)

    # ---- forward -------------------------------------------------------------------------------------------
    def forward(self, ycat: torch.Tensor, nreal: int):
        """ycat fp32 [2B, T]: rows [0, nreal) real, the rest generated.  Weight-norm sub-discriminators run the
        whole batch through each layer once; the spectral-norm one runs the two halves with their own weights,
        because the reference's d(y) and d(y_hat) calls each advance the power iteration (models.py:236-244)."""
        L = _lib.lib()
        nb, t = ycat.shape
        G = self._geometry(nb, t)
        period = self.period
        parts = [(0, nb)] if not self.spectral else [(0, nreal), (nreal, nb - nreal)]
        self.parts = []
        # weight_norm layers: the packs stay valid until the next optimizer update (the G-step forward of one step
        # and the D-step forward of the next see the same weights); spectral norm moves on every call, and its
        # second part's power iteration continues from the first's.  The layers are independent of each other, so
        # their fold / power-iteration / pack chains are spread over the prep lanes (part 0 before part 1 per layer).
        if self.spectral and self._prefetched is not None:
            # prefetch_weights() queued this call's power iterations and forward banks on the prep lanes
            Ws, self._prefetched = self._prefetched, None
            torch.cuda.current_stream().wait_stream(self.prep.streams[0])
            self.W_cached = Ws[-1]
            self.fwd_valid = True
        elif self.spectral or not self.fwd_valid:
            if self.spectral:
                # the power iterations of the layers are independent chains of three small kernels (part 0 before part 1
                # per layer: the second call continues from the first's u, v): side by side on the prep lanes.  (Batched
                # per stage over all layers, or as one cluster launch, they were slower: a many-block launch on this
                # lane waits for whole tensor-core kernels of the other lanes to drain — profiles/r02_summary.md.)
                Ws = [self._weights(pi) for pi in range(len(parts))]
                self.prep.fork()
                for li in range(len(self.mods)):
                    with self.prep.lane(li):
                        for pi, W in enumerate(Ws):
                            self._weights_layer(W, self.wbufs[pi], li)
                self.prep.join()
                for pi in range(len(parts)):
                    self._table(pi).launch("fwd")
            else:
                Ws = [self._prepare_weights(0)]
            self.W_cached = Ws[-1]
            self.fwd_valid = True
        else:
            Ws = [self.W_cached]
        here = torch.cuda.current_stream()
        # the data-gradient filter banks of these weights: one batched launch per part, on a high-priority lane beside
        # the forward chain (on the low-priority w-lane a many-block launch starves behind the other lanes' tensor-core
        # kernels and holds the backward up); the backward waits for it before its first data-gradient launch
        plane = self.prep.streams[0]
        plane.wait_stream(here)
        with torch.cuda.stream(plane):
            for pi in range(len(parts)):
                self._pack_dgrad(Ws[pi], pi)
        if len(parts) > 1:
            # the second part's chain forks HERE, before the first part's launches are queued on this stream: the
            # two halves run side by side (they wrote "wait_stream(here)" after part 0 once, and ran one after the
            # other: 300 us of the step's critical path per forward — profiles/r02_summary.md section 2)
            self.lanes.streams[1].wait_stream(here)
        for pi, (b0, bn) in enumerate(parts):
            W = Ws[pi]
            self.parts.append((b0, bn, W))
            if pi == 1:
                with torch.cuda.stream(self.lanes.streams[1]):
                    self._forward_part(L, G, W, ycat, b0, bn, t)
            else:
                self._forward_part(L, G, W, ycat, b0, bn, t)
        if len(parts) > 1:
            here.wait_stream(self.lanes.streams[1])
        self.G, self.nb, self.nreal, self.t, self.ycat = G, nb, nreal, t, ycat
        return G

    def _forward_part(self, L, G, W, ycat, b0: int, bn: int, t: int) -> None:
        period = self.period
        st = _stream()
        k0, s0, p0, c0 = self.first
        seq0, nseq = b0 * period, bn * period
        w0 = W["eff"][0].reshape(c0, k0).contiguous()
        W["w0"] = w0
        b0_bias = self.mods[0].bias
        act = G["act"][0]
        h, rows, _ = G["geo"][0]
        _lib.check(L.hg_disc_first_conv_fwd(ycat[b0:].data_ptr(), w0.data_ptr(), b0_bias.data_ptr(), bn, t, period,
                                            k0, s0, p0, c0, rows, act[seq0:].data_ptr(), LRELU_SLOPE, st),
                   "hg_disc_first_conv_fwd")
        for li, layer in enumerate(self.mids):
            m = self.mods[1 + li]
            bias = m.bias
            out = G["act"][1 + li]
            h_out, rows_out, _ = G["geo"][1 + li]
            _lib.check(L.hg_conv1d_general_fwd(act[seq0:].data_ptr(), W["fwd"][1 + li].data_ptr(), bias.data_ptr(),
                                               1, nseq * rows, layer.cin, nseq * rows_out, nseq * rows_out,
                                               layer.groups_eff, layer.cout, layer.k, layer.stride, layer.pad,
                                               out[seq0:].data_ptr(), LRELU_SLOPE, 0, rows_out, h_out, st),
                       "hg_conv1d_general_fwd")
            act, h, rows = out, h_out, rows_out
        c_last = G["geo"][-1][2]
        wp = W["eff"][-1].reshape(c_last, self.kpost).contiguous()
        W["wp"] = wp
        bp = self.mods[-1].bias
        _lib.check(L.hg_disc_last_conv_fwd(act[seq0:].data_ptr(), wp.data_ptr(), bp.data_ptr(), nseq, h, rows,
                                           c_last, self.kpost, G["logit"][seq0:].data_ptr(), st),
                   "hg_disc_last_conv_fwd")

    # ---- losses (on the internal layouts; means are permutation-invariant) -------------------------------------
    def numel_fmaps(self, nb_half: int) -> List[int]:
        """element counts of the reference's feature maps for a batch of nb_half items"""
        return [nb_half * self.period * h * c for h, _, c in self.G["geo"]] + [nb_half * self.period * self.G["geo"][-1][0]]

    def loss_terms(self, acc: torch.Tensor, slot: int, fm: bool = True) -> None:
        """acc[slot + 0] += sum (1 - logit_r)^2, [1] += sum logit_g^2, [2] += sum (1 - logit_g)^2,
        acc[slot + 3 + l] += sum |fmap_r[l] - fmap_g[l]| (l = 0..n_layers, the last one the logits) — every
        reduction of this sub-discriminator in ONE launch (a HG_JOB_LOSS_SUM job table per geometry)."""
        G, period = self.G, self.period
        nr = self.nreal * period
        ng = (self.nb - self.nreal) * period
        fm = fm and nr == ng           # feature-matching sums: only the generator step reads them
        key = ("loss", acc.data_ptr(), slot, fm, nr, ng)
        tab = G.get(key)
        if tab is None:
            from . import batched
            tab = batched.JobTable(self.device)
            h = G["geo"][-1][0]
            lr, lg = G["logit"][:nr], G["logit"][nr:]
            out = lambda i: acc.data_ptr() + 4 * (slot + i)
            tab.add_loss_sum("sum", 1, lr, None, nr * h, 1.0, out(0))
            tab.add_loss_sum("sum", 1, lg, None, ng * h, 0.0, out(1))
            tab.add_loss_sum("sum", 1, lg, None, ng * h, 1.0, out(2))
            if fm:
                for l, a in enumerate(G["act"]):
                    n = a[:nr].numel()
                    if n % 8:
                        raise RuntimeError("feature map size must be a multiple of 8 elements")
                    tab.add_loss_sum("sum", 2, a, a[nr:], n // 8, 0.0, out(3 + l), chunk=4096)
                tab.add_loss_sum("sum", 0, lr, lg, nr * h, 0.0, out(3 + len(G["act"])))
            G[key] = tab.finalize()
        tab.launch("sum")

    # ---- backward ------------------------------------------------------------------------------------------
    def backward_d(self) -> None:
        """discriminator step: d loss_disc / d parameters, both halves (full dgrad + wgrad)."""
        L = _lib.lib()
        G, period, st = self.G, self.period, _stream()
        nr = self.nreal * period
        ntot = self.nb * period
        h = G["geo"][-1][0]
        lr, lg = G["logit"][:nr], G["logit"][nr:]
        # d/dlogit of mean((1 - lr)^2) + mean(lg^2)
        _lib.check(L.hg_loss_grad(lr.data_ptr(), 0, nr * h, 1, 1.0, 2.0 / (nr * h), 0.0, 0, G["dlogit"].data_ptr(), st))
        _lib.check(L.hg_loss_grad(lg.data_ptr(), 0, (ntot - nr) * h, 1, 0.0, 2.0 / ((ntot - nr) * h), 0.0, 0,
                                  G["dlogit"][nr:].data_ptr(), st))
        here = torch.cuda.current_stream()
        here.wait_stream(self.prep.streams[0])      # data-gradient packs (queued by forward on the pack lane)
        if not self.spectral:
            self.dwp_flat.zero_()
        self.lanes.fork()     # both lanes join the capture here (a join of a never-forked stream would invalidate it)
        self.wl.fork()
        for pi, (b0, bn, W) in enumerate(self.parts):
            if pi == 1:                       # spectral norm: the generated half's chain on the second lane,
                with torch.cuda.stream(self.lanes.streams[1]):     # beside the real half's (forked just above)
                    self._backward_part(L, G, W, b0, bn, want_wgrad=True, fm=False, dy_audio=None, accumulate=True,
                                        part=pi)
            else:
                self._backward_part(L, G, W, b0, bn, want_wgrad=True, fm=False, dy_audio=None, accumulate=True,
                                    part=pi)
        self.wl.join()
        self.lanes.join()

    def _bwd_bank(self, part: int):
        """data-gradient filter banks of part / call slot `part` (created on first use)"""
        while len(self.bwd_parts) <= part:
            self.bwd_parts.append([_DiscBwdLayer(l, self.device) for l in self.mids])
        return self.bwd_parts[part]

    def _pack_dgrad(self, W, part: int = 0) -> None:
        if self.spectral or not self.dgrad_valid:
            t = self._table(part)
            if t.has("dgrad"):
                t.launch("dgrad")
            for i in self.untiled:
                self._bwd_bank(part)[i].pack(W["eff"][1 + i])
            self.dgrad_valid = True

    # ---- one module call under torch autograd (autograd.py): forward with its own activation / weight slot ---------
    def forward_single(self, x2d: torch.Tensor, slot: int, dgrad: bool = True):
        """x2d fp32 [B, T] -> (G, W) of call slot `slot`: activations, logits, the weights this call used (a train-mode
        spectral-norm layer advances its power iteration per call, like the reference's hook) and, with `dgrad`
        (the call can be differentiated), their data-gradient banks.  Everything on the current stream."""
        L = _lib.lib()
        nb, t = x2d.shape
        G = self._geometry(nb, t, slot)
        W = self._prepare_weights(slot)
        if dgrad:
            tb = self._table(slot)
            if tb.has("dgrad"):
                tb.launch("dgrad")
            for i in self.untiled:
                self._bwd_bank(slot)[i].pack(W["eff"][1 + i])
        self._forward_part(L, G, W, x2d, 0, nb, t)
        return G, W

    def backward_single(self, G, W, slot: int, x2d: torch.Tensor, dlogit: torch.Tensor, pre_adds, want_wgrad: bool,
                        dy_audio) -> None:
        """Backward of forward_single's call: dlogit fp32 [B*period][h] (internal order), pre_adds[l] bf16 gradient at
        feature map l in the internal layout (or None) -> parameter gradients ADDED into self.flat (want_wgrad)
        and / or the audio gradient ADDED into dy_audio fp32 [B][T]."""
        L = _lib.lib()
        nb, t = x2d.shape
        self.G, self.nb, self.nreal, self.t, self.ycat = G, nb, nb, t, x2d
        G["dlogit"].copy_(dlogit)
        if want_wgrad and not self.spectral:
            self.dwp_flat.zero_()
        self.lanes.fork()
        self.wl.fork()
        self._backward_part(L, G, W, 0, nb, want_wgrad=want_wgrad, fm=False, dy_audio=dy_audio, accumulate=True,
                            part=slot, pre_adds=pre_adds)
        self.wl.join()
        self.lanes.join()

    def backward_g(self, dy_audio: torch.Tensor, nfm: List[float]) -> None:
        """generator step: d (loss_gen + loss_fm) / d y_g_hat accumulated into dy_audio fp32 [B][T] (generated half
        only, no weight gradients).  nfm[l] = 2 / numel(fmap l) (feature_loss doubles the sum of means)."""
        L = _lib.lib()
        G, period, st = self.G, self.period, _stream()
        nr = self.nreal * period
        ng = (self.nb - self.nreal) * period
        h = G["geo"][-1][0]
        lr, lg = G["logit"][:nr], G["logit"][nr:]
        # d/dlg of mean((1 - lg)^2) + 2 * mean|lr - lg|
        _lib.check(L.hg_loss_grad(lg.data_ptr(), lr.data_ptr(), ng * h, 2, 1.0, 2.0 / (ng * h), nfm[-1], 0,
                                  G["dlogit"][nr:].data_ptr(), st))
        b0, bn, W = self.parts[-1] if self.spectral else (self.nreal, self.nb - self.nreal, self.parts[0][2])
        part = len(self.parts) - 1
        torch.cuda.current_stream().wait_stream(self.prep.streams[0])     # data-gradient packs (see forward)
        self._backward_part(L, G, W, self.nreal, self.nb - self.nreal, want_wgrad=False, fm=True,
                            dy_audio=dy_audio, accumulate=False, nfm=nfm, part=part)

    def _backward_part(self, L, G, W, b0: int, bn: int, want_wgrad: bool, fm: bool, dy_audio, accumulate: bool,
                       nfm: Optional[List[float]] = None, part: int = 0, pre_adds=None) -> None:
        """The data-gradient chain runs on the current stream; all parameter-gradient work (bias sums, wgrad,
        finish) goes to this sub-discriminator's w-lane, which also serialises the use of the shared scratch."""
        period = self.period
        seq0, nseq = b0 * period, bn * period
        nr = self.nreal * period
        geo = G["geo"]
        nl = len(self.mids)
        bwd = self._bwd_bank(part)
        pre = pre_adds if pre_adds is not None else [None] * (nl + 1)   # incoming feature-map gradients (autograd path)
        h_last, rows_last, c_last = geo[-1]
        act_last = G["act"][-1]
        post = self.mods[-1]
        here = torch.cuda.current_stream()

        def side(fn, chain: int):
            # chain c (one layer's parameter gradients) runs on lane c % n_chains with a scratch of its own; the two
            # halves of a spectral-norm layer use the same lane, so their accumulation into the layer's gradient
            # stays ordered
            wlane = self.wl.streams[chain % self.n_chains]
            wlane.wait_stream(here)
            with torch.cuda.stream(wlane):
                fn(self._scratch_of(chain))

        # fm_r for the generated half is the real half of the same buffer (seq - nr)
        fm_r_last = act_last[seq0 - nr:].data_ptr() if fm else 0
        # every data-gradient launch of the discriminator step also sums the bias gradient of the layer whose output
        # it differentiates, in fp32, straight into the flat gradient buffer (zeroed in run_phases)
        bias_of = (lambda li: self.flat.grad(self.mods[li].bias).data_ptr()) if want_wgrad else (lambda li: 0)
        _lib.check(L.hg_disc_last_conv_bwd(act_last[seq0:].data_ptr(), W["wp"].data_ptr(), G["dlogit"][seq0:].data_ptr(),
                                           nseq, h_last, rows_last, c_last, self.kpost, LRELU_SLOPE, fm_r_last,
                                           nfm[nl] if fm else 0.0, _p(pre[nl]), G["grad"][-1][seq0:].data_ptr(), 0, 0,
                                           bias_of(nl), _stream()), "hg_disc_last_conv_bwd")
        if want_wgrad:
            def post_grads(scratch):
                scratch[: c_last * self.kpost].zero_()
                self.db.zero_()
                _lib.check(L.hg_disc_last_conv_bwd(act_last[seq0:].data_ptr(), W["wp"].data_ptr(),
                                                   G["dlogit"][seq0:].data_ptr(), nseq, h_last, rows_last, c_last,
                                                   self.kpost, LRELU_SLOPE, 0, 0.0, 0, 0, scratch.data_ptr(),
                                                   self.db.data_ptr(), 0, _stream()), "hg_disc_last_conv_bwd")
                self._route(L, post, scratch, 1, c_last * self.kpost, W, len(self.mods) - 1, True)
                self._bias(post, self.db[:1], True)
            side(post_grads, 0)
        for li in reversed(range(nl)):
            layer = self.mids[li]
            m = self.mods[1 + li]
            h_out, rows_out, _ = geo[1 + li]
            h_in, rows_in, c_in = geo[li]
            d_out = G["grad"][1 + li][seq0:]
            a_in = G["act"][li]
            if want_wgrad:
                def layer_grads(scratch, layer=layer, m=m, li=li, h_out=h_out, rows_out=rows_out, rows_in=rows_in,
                                d_out=d_out, a_in=a_in):
                    st = _stream()
                    sn = hasattr(m, "weight_orig")
                    # weight_norm layers: dwps[li] was zeroed with the whole region (zero_wgrads) and is finished by
                    # hg_wgrad_finish_conv below; the spectral-norm scale's two halves each need their own sigma, so
                    # they start from zero and are routed layer by layer
                    _lib.check(L.hg_conv1d_wgrad(a_in[seq0:].data_ptr(), d_out.data_ptr(), 1, nseq * rows_in, layer.cin,
                                                 nseq * rows_out, nseq * rows_out, layer.groups_eff, layer.cout,
                                                 layer.k, layer.stride, 1, layer.pad, self.dwps[li].data_ptr(),
                                                 0 if sn else 1, st), "hg_conv1d_wgrad")
                    cin_g = layer.cin // layer.groups
                    order = (c_int * layer.k)(*layer.order)
                    if sn:
                        _lib.check(L.hg_unpack_wgrad_conv(self.dwps[li].data_ptr(), layer.cout, cin_g, layer.k,
                                                          layer.cout, layer.cin_tile, layer.cout // layer.groups,
                                                          layer.merge, order, scratch.data_ptr(), st),
                                   "hg_unpack_wgrad_conv")
                        self._route(L, m, scratch, layer.cout, cin_g * layer.k, W, 1 + li, True)
                    else:
                        g, v = _g_v(m)          # unpack + weight_norm backward in one launch, accumulating
                        _lib.check(L.hg_wgrad_finish_conv(self.dwps[li].data_ptr(), layer.cout, cin_g, layer.k,
                                                          layer.cout, layer.cin_tile, layer.cout // layer.groups,
                                                          layer.merge, order, v.data_ptr(), g.data_ptr(), 1,
                                                          self.flat.grad(v).data_ptr(), self.flat.grad(g).data_ptr(),
                                                          st), "hg_wgrad_finish_conv")
                side(layer_grads, nl - li)
            bwd[li].dgrad(L, d_out, nseq, h_out, rows_out, rows_in, a_in[seq0:],
                          a_in[seq0 - nr:] if fm else None, nfm[li] if fm else 0.0, G["grad"][li][seq0:], _stream(),
                          flat_h_in=h_in, bias_dst=bias_of(li), pre_add=pre[li])
        # first conv (Cin = 1)
        k0, s0, p0, c0 = self.first
        m0 = self.mods[0]
        if want_wgrad:
            def first_grads(scratch):
                scratch[: c0 * k0].zero_()
                # the kernel's own bias column (summed from the bf16 gradient) lands in the db scratch and is not
                # used: the first conv's bias gradient came from the fp32 sums of the launch that produced grad[0]
                _lib.check(L.hg_disc_first_conv_bwd(self.ycat[b0:].data_ptr(), W["w0"].data_ptr(),
                                                    G["grad"][0][seq0:].data_ptr(), bn, self.t, period, k0, s0, p0, c0,
                                                    geo[0][1], scratch.data_ptr(), self.db_unused.data_ptr(), 0,
                                                    _stream()), "hg_disc_first_conv_bwd")
                self._route(L, m0, scratch, c0, k0, W, 0, True)
            side(first_grads, nl + 1)
        if dy_audio is not None:
            _lib.check(L.hg_disc_first_conv_bwd(self.ycat[b0:].data_ptr(), W["w0"].data_ptr(),
                                                G["grad"][0][seq0:].data_ptr(), bn, self.t, period, k0, s0, p0, c0,
                                                geo[0][1], 0, 0, _p(dy_audio), _stream()), "hg_disc_first_conv_bwd")

    def _bias(self, m: nn.Module, db: torch.Tensor, accumulate: bool) -> None:
        if accumulate:
            self.flat.grad(m.bias).add_(db)
        else:
            self.flat.grad(m.bias).copy_(db)

    def _route(self, L, m: nn.Module, dw: torch.Tensor, d0: int, rest: int, W, li: int, accumulate: bool) -> None:
        if hasattr(m, "weight_orig"):
            # spectral norm: w = W / sigma with sigma = u^T W v (u, v constants): dW = (dw - <dw, w> u v^T) / sigma
            u, v, sigma, snws = W["sn"][li]
            _lib.check(L.hg_spectral_norm_bwd(dw.data_ptr(), W["eff"][li].data_ptr(), u.data_ptr(), v.data_ptr(),
                                              sigma.data_ptr(), d0, rest, 1 if accumulate else 0,
                                              self.flat.grad(m.weight_orig).data_ptr(), snws.data_ptr(), _stream()),
                       "hg_spectral_norm_bwd")
        else:
            _route_weight_grad(L, self.flat, m, dw, d0, rest, accumulate)


class DiscriminatorTrainer:
    """MultiPeriodDiscriminator + MultiScaleDiscriminator of one training step."""

    def __init__(self, mpd: MultiPeriodDiscriminator, msd: MultiScaleDiscriminator, device):
        self.mpd, self.msd, self.device = mpd, msd, device
        holder = nn.ModuleList([mpd, msd])        # optimizer order of the reference: chain(msd, mpd) — order is free
        self.flat = FlatParams(holder, device)
        # scheduling: the scale discriminators' chains (k = 41 grouped convs, spectral norm) are long and narrow, the
        # period discriminators' short and wide; the scales' lanes outrank the periods' so that they are done by the
        # time the periods fill the GPU (HG_DISC_BOOST="a,b,c" sets the three boosts, "0" disables; measured
        # -2,-1,-1: 11.86 ms, 0,0,0: 11.98, -2,-1,0: 12.12, -2,-2,-2: 12.9 in round 2)
        env = os.environ.get("HG_DISC_BOOST", "")
        boosts = [0, 0, 0] if env == "0" else [int(v) for v in env.split(",")] if "," in env else [-2, -1, -1]
        self.subs_p = [_SubDiscTrainer(d, device, self.flat) for d in mpd.discriminators]
        self.subs_s = [_SubDiscTrainer(d, device, self.flat, boosts[min(i, 2)])
                       for i, d in enumerate(msd.discriminators)]
        self.subs = self.subs_p + self.subs_s
        self.nslots = 12
        # raw loss sums of the discriminator-step forward / of the generator-step forward
        self.acc_d = torch.zeros(len(self.subs) * self.nslots, dtype=torch.float32, device=device)
        self.acc_g = torch.zeros_like(self.acc_d)
        self.pooled: List[torch.Tensor] = []
        self._inv_counts: Dict[Tuple[int, int], torch.Tensor] = {}
        self.lanes = _Lanes(len(self.subs), device,                          # one per sub-discriminator
                            [-1] * len(self.subs_p) + [-1 + boosts[min(i, 2)] for i in range(len(self.subs_s))])
        self.spans = [self.flat.span_of(d) for d in list(mpd.discriminators) + list(msd.discriminators)]
        self.order = list(range(len(self.subs)))
        self.order_fixed = False                          # True once measured (TrainStep.step_graphed) or forced
        forced = os.environ.get("HG_LANE_ORDER")          # e.g. "6,4,0,3,2,1,7,5": experiments (same on every rank!)
        if forced:
            self.order = [int(v) for v in forced.split(",")]
            if sorted(self.order) != list(range(len(self.subs))):
                raise ValueError("HG_LANE_ORDER must be a permutation of the sub-discriminator indices")
            self.order_fixed = True
        if self.spans[0][0] != 0 or self.spans[-1][1] != self.flat.numel or any(
                a[1] != b[0] for a, b in zip(self.spans, self.spans[1:])):
            raise RuntimeError("DiscriminatorTrainer: sub-discriminator parameter spans do not tile the flat buffer")

    def _inputs(self, y: torch.Tensor, y_hat: torch.Tensor) -> int:
        """(real ++ generated) audio and its AvgPool1d(4,2,2) pyramid for the scale discriminators"""
        b = y.shape[0]
        ycat = torch.cat([y.reshape(b, -1), y_hat.reshape(b, -1)], 0).contiguous().float()
        self.b, self.t = b, ycat.shape[1]
        self.pooled = [ycat]
        for i in range(1, len(self.subs_s)):
            self.pooled.append(_avgpool(self.pooled[-1]))
        return b

    def _input_of(self, i: int) -> torch.Tensor:
        return self.pooled[0] if i < len(self.subs_p) else self.pooled[i - len(self.subs_p)]

    def run_phases(self, y: torch.Tensor, y_hat: torch.Tensor, dy_audio: torch.Tensor, update: bool, lr: float, betas,
                   world: int = 1, allreduce=None, stamps: Optional[LaneStamps] = None
                   ) -> Tuple[Dict[str, torch.Tensor], Dict[str, torch.Tensor]]:
        """The discriminator step and the discriminator half of the generator step of ONE training step, with every
        sub-discriminator running its whole chain on its own lane:
            forward -> loss sums -> backward (parameter gradients) -> AdamW on its own slice of the flat buffers
            -> forward with the updated weights -> loss sums -> data gradient into dy_audio.
        The lanes only meet at the end, so a short chain (a period discriminator) is already in its generator-step
        forward while the longest one (the spectral-norm scale) is still in its backward; data-parallel, each lane
        all-reduces its own gradient slice between its backward and its AdamW.  Same arithmetic as forward / backward_d / adamw / forward / backward_g in sequence.
        Returns (discriminator-step losses, generator-step losses); dy_audio fp32 [B][T] is ADDED to."""
        L = _lib.lib()
        b = self._inputs(y, y_hat)
        self.acc_d.zero_()
        self.acc_g.zero_()
        self.flat.g.zero_()                 # every parameter-gradient kernel of the sub-discriminators accumulates
        guard = update and self.flat.guarded
        if update and not guard:
            self.flat.bump_step()
        grads = [dy_audio] + [torch.zeros(b, p.shape[1], dtype=torch.float32, device=self.device)
                              for p in self.pooled[1:]]
        np_ = len(self.subs_p)
        mark = stamps.mark if stamps is not None else (lambda name: None)
        self.lanes.fork()
        # Python issue order = the order of the slices on NCCL's (single, in-order) stream: a slice queued behind the
        # slice of a lane that finishes its backward later waits for it.  self.order lists the lanes by the time
        # their backward ends in the replayed step (measured: tests/lane_stamps.py).
        for i in self.order:
            sd = self.subs[i]
            with self.lanes.lane(i):
                sd.forward(self._input_of(i), b)
                sd.loss_terms(self.acc_d, i * self.nslots, fm=False)
                sd.backward_d()
                mark(f"d{i}_bwd_done")
                if world > 1:
                    # this sub-discriminator's slice of the gradient buffer, exchanged as soon as its backward is
                    # done: the collectives run in issue order on NCCL's stream while the later lanes still compute
                    allreduce(self.flat, self.spans[i])
                    mark(f"d{i}_allreduce_done")
                if guard:
                    self.flat.grad_norm(i, *self.spans[i])     # slot = sub-discriminator: a fixed summation order
        if guard:
            # the norm is global over every slice: the lanes meet once every gradient is final (the barrier torch's
            # clip_grad_norm_ over optim_d's parameters implies), then fork again for the updates
            self.lanes.join()
            self.flat.finalize_norm(1.0 / world)
            self.lanes.fork()
        for i in self.order:
            sd = self.subs[i]
            with self.lanes.lane(i):
                if update:
                    self.flat.adamw_slice(self.spans[i][0], self.spans[i][1], lr, betas, grad_scale=1.0 / world)
                    sd.invalidate()
                sd.forward(self._input_of(i), b)
                sd.loss_terms(self.acc_g, i * self.nslots)
                sd.backward_g(grads[0] if i < np_ else grads[i - np_], [2.0 / n for n in sd.numel_fmaps(b)])
                mark(f"d{i}_gstep_done")
        self.lanes.join()
        for i in reversed(range(1, len(grads))):
            _lib.check(L.hg_avgpool_4_2_2_bwd(grads[i].data_ptr(), b, grads[i - 1].shape[1], grads[i - 1].data_ptr(),
                                              _stream()), "hg_avgpool_4_2_2_bwd")
        return self.losses(self.acc_d), self.losses(self.acc_g)

    def losses(self, acc: torch.Tensor) -> Dict[str, torch.Tensor]:
        """loss values from the accumulated sums of one forward (device tensors, no host sync)."""
        a = acc.view(len(self.subs), self.nslots)
        out = {}
        np_ = len(self.subs_p)
        key = (self.b, self.t)
        inv = self._inv_counts.get(key)
        if inv is None:
            # 1 / numel of every loss term, laid out like self.acc (slots 0-2: logits, 3..: feature maps, x2)
            host = torch.zeros(len(self.subs), self.nslots)
            for i, sd in enumerate(self.subs):
                n = sd.numel_fmaps(self.b)
                host[i, 0:3] = 1.0 / n[-1]
                host[i, 3:3 + len(n)] = 2.0 / torch.tensor(n, dtype=torch.float64)
            inv = host.to(self.device)
            self._inv_counts[key] = inv
        terms = a * inv
        out["loss_disc_f"], out["loss_disc_s"] = terms[:np_, 0:2].sum(), terms[np_:, 0:2].sum()
        out["loss_gen_f"], out["loss_gen_s"] = terms[:np_, 2].sum(), terms[np_:, 2].sum()
        out["loss_fm_f"], out["loss_fm_s"] = terms[:np_, 3:].sum(), terms[np_:, 3:].sum()
        return out


# ------------------------------------------------------------------------------------------------ the step
class TrainStep:
    """One process's share of the UPSTREAM train loop body.  With torch.distributed initialised (NCCL, one process
    per GPU) the flat gradient buffers are all-reduced (sum) after each backward and AdamW divides by world size —
    identical to DistributedDataParallel's gradient averaging."""

    def __init__(self, generator: Generator, mpd: MultiPeriodDiscriminator, msd: MultiScaleDiscriminator, h,
                 device=None, process_group=None):
        device = torch.device(device if device is not None else "cuda")
        self.h, self.device = h, device
        generator.to(device); mpd.to(device); msd.to(device)
        generator.train(); mpd.train(); msd.train()
        self.G = GeneratorTrainer(generator, device)
        self.D = DiscriminatorTrainer(mpd, msd, device)
        self.lr = h.learning_rate
        self.betas = (h.adam_b1, h.adam_b2)
        self.pg = process_group
        self.mel_lane = torch.cuda.Stream(device=device)
        self.capture_stream = torch.cuda.Stream(device=device, priority=-1)
        self.world = 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            self.world = torch.distributed.get_world_size(process_group)
        self.stamps = LaneStamps(device)
        # h.clip_grad_norm (optional; null / absent = off): each network's update follows the fork's callback,
        # total = clip_grad_norm_(params, clip_grad_norm); optim.step() only if total is finite
        self.clip_grad_norm = getattr(h, "clip_grad_norm", None)
        if self.clip_grad_norm is not None:
            self.G.flat.enable_guard(self.clip_grad_norm)
            self.D.flat.enable_guard(self.clip_grad_norm, slots=len(self.D.subs))

    def _allreduce(self, flat: FlatParams, span: Optional[Tuple[int, int]] = None) -> None:
        allreduce_gradients(flat, self.pg, span)

    def _mel_plan(self):
        """the loss-mel plan (fmax_for_loss), created through the public function's cache"""
        h = self.h
        dev = self.G.flat.p.device          # the resolved device ("cuda:0"), as mel_spectrogram spells its cache key
        key = (f'{str(dev)}_{h.n_fft}_{h.num_mels}_{h.sampling_rate}_{h.hop_size}_{h.win_size}_{h.fmin}_'
               f'{h.fmax_for_loss}_False')
        plan = torch_mels.get(key)
        if plan is None:
            mel_spectrogram(torch.zeros(1, h.segment_size, device=self.device), h.n_fft, h.num_mels, h.sampling_rate,
                            h.hop_size, h.win_size, h.fmin, h.fmax_for_loss)
            plan = torch_mels[key]
        return plan

    def step(self, x: torch.Tensor, y: torch.Tensor, y_mel: torch.Tensor, update: bool = True) -> Dict[str, torch.Tensor]:
        """x [B,80,F] input mel, y [B,1,T] audio, y_mel [B,80,F] loss mel.  Returns the loss tensors (device)."""
        L = _lib.lib()
        h = self.h
        b = x.shape[0]
        st = _stream()
        if not torch.cuda.is_current_stream_capturing():
            self.G.flat.set_lr(self.lr)
            self.D.flat.set_lr(self.lr)
        launches0 = _lib.launch_count()
        self.stamps.begin()
        self.stamps.mark("start")
        y2 = y.reshape(b, -1).contiguous().float()
        for sd in self.D.subs:
            sd.prefetch_weights()                              # spectral-norm weights of the D step, beside G's forward
        y_g = self.G.forward(x)                                # [B,1,T]
        y_g2 = y_g.view(b, -1)
        out: Dict[str, torch.Tensor] = {}
        # ---- mel loss of the generated audio and its gradient: its own lane, beside the discriminator work
        plan = self._mel_plan()
        n_frames = plan.frames(y_g2.shape[1])
        mel_g = torch.empty(b, h.num_mels, n_frames, dtype=torch.float32, device=self.device)
        n_mel = mel_g.numel()
        acc = torch.zeros(1, dtype=torch.float32, device=self.device)
        ym = y_mel.contiguous().float()
        dmel = torch.empty_like(mel_g)
        dy = torch.zeros(b, y_g2.shape[1], dtype=torch.float32, device=self.device)   # every producer ADDS into it
        here = torch.cuda.current_stream()
        self.mel_lane.wait_stream(here)
        with torch.cuda.stream(self.mel_lane):
            ms = _stream()
            _lib.check(L.hg_mel_fwd(plan.handle, y_g2.data_ptr(), b, y_g2.shape[1], mel_g.data_ptr(), 0, ms), "hg_mel_fwd")
            _lib.check(L.hg_loss_sum(ym.data_ptr(), mel_g.data_ptr(), n_mel, 0, 0.0, acc.data_ptr(), ms), "hg_loss_sum")
            _lib.check(L.hg_loss_grad(mel_g.data_ptr(), ym.data_ptr(), n_mel, 0, 0.0, 45.0 / n_mel, 0.0, 0,
                                      dmel.data_ptr(), ms), "hg_loss_grad")
            _lib.check(L.hg_mel_bwd(plan.handle, y_g2.data_ptr(), dmel.data_ptr(), b, y_g2.shape[1], dy.data_ptr(), ms),
                       "hg_mel_bwd")
        # ---- discriminator step, then the generator step's pass through the updated discriminators
        self.stamps.mark("g_fwd_done")
        dl, gl = self.D.run_phases(y2, y_g2, dy, update, self.lr, self.betas, self.world, self._allreduce, self.stamps)
        here.wait_stream(self.mel_lane)
        out["loss_mel"] = acc[0] / n_mel * 45
        out["loss_disc_f"], out["loss_disc_s"] = dl["loss_disc_f"], dl["loss_disc_s"]
        out["loss_disc_all"] = dl["loss_disc_f"] + dl["loss_disc_s"]
        for k in ("loss_gen_f", "loss_gen_s", "loss_fm_f", "loss_fm_s"):
            out[k] = gl[k]
        out["loss_gen_all"] = gl["loss_gen_s"] + gl["loss_gen_f"] + gl["loss_fm_s"] + gl["loss_fm_f"] + out["loss_mel"]
        self.dy_audio = dy
        self.stamps.mark("g_bwd_start")
        self.G.backward(dy)
        self.stamps.mark("g_bwd_done")
        self._allreduce(self.G.flat)
        self.stamps.mark("g_allreduce_done")
        if update:
            if self.G.flat.guarded:
                self.G.flat.grad_norm()
                self.G.flat.finalize_norm(1.0 / self.world)
            self.G.flat.adamw(self.lr, self.betas, grad_scale=1.0 / self.world)
            self.G.invalidate()
        self.stamps.mark("end")
        out["y_g_hat"] = y_g
        if self.clip_grad_norm is not None:
            # static device buffers (refreshed by every step and graph replay): read them before the next step
            for name, flat in (("g", self.G.flat), ("d", self.D.flat)):
                out[f"grad_norm_{name}"] = flat.grad_norm_dev[0]
                out[f"skipped_steps_{name}"] = flat.skipped_dev[0]
        self.launches_per_step = _lib.launch_count() - launches0   # library kernels issued (or captured) per step
        return out

    @property
    def graph_active(self) -> bool:
        return any(isinstance(v, list) for v in self.__dict__.get("_graphs", {}).values())

    # ---- CUDA-graph replay ---------------------------------------------------------------------------------------
    def step_graphed(self, x: torch.Tensor, y: torch.Tensor, y_mel: torch.Tensor) -> Dict[str, torch.Tensor]:
        """`step` replayed as ONE CUDA graph (about 3000 launches per step are otherwise host-bound at batch 16).
        The first call of a shape runs eagerly (it is a real step and loads every kernel); the second call captures
        and replays; later calls copy the inputs into the captured buffers and replay.  The returned loss tensors are
        the graph's static outputs: read them before the next call.  Falls back to eager when capture fails."""
        self.G.flat.set_lr(self.lr)
        self.D.flat.set_lr(self.lr)
        key = (tuple(x.shape), tuple(y.shape), self.world)
        graphs = self.__dict__.setdefault("_graphs", {})
        entry = graphs.get(key)
        if entry is None:
            graphs[key] = "seen"
            return self.step(x, y, y_mel)
        calibrate = self.world > 1 and not self.D.order_fixed
        if isinstance(entry, list) and calibrate and entry[5] >= self.CALIBRATION_REPLAYS:
            self._calibrate_slice_order()
            calibrate = not self.D.order_fixed      # another round (marks stay on) or the final capture (marks off)
            entry = graphs[key] = "seen"            # capture again below with the slices in the new order
        if entry == "seen":
            sx, sy, sm = x.clone(), y.clone(), y_mel.clone()
            torch.cuda.synchronize()
            # The captured step must not depend on host cache state: anything that refreshed the generator's packs
            # since the last update (a validation `generator(x)` between the eager and the capture step) would make
            # every refresh a host-side no-op here and the graph would replay G on stale bf16 weights for ever.
            self.G.invalidate()
            self.stamps.force = calibrate           # the first data-parallel capture carries the lane time marks
            try:
                g = torch.cuda.CUDAGraph()
                # thread_local: the NCCL watchdog thread of a data-parallel run may touch the CUDA API meanwhile
                # captured on a high-priority stream: the main chain (generator forward / data gradients) outranks
                # the parameter-gradient lanes
                with torch.cuda.graph(g, stream=self.capture_stream, capture_error_mode="thread_local"):
                    out = self.step(sx, sy, sm)
                entry = [g, sx, sy, sm, out, 0]
            except Exception as e:  # noqa: BLE001
                import warnings
                warnings.warn(f"hifigan_b200: CUDA graph capture of the training step failed, running eagerly ({e})")
                torch.cuda.synchronize()
                entry = "eager"
                # the aborted capture ran the host side of a step (flags, caches) without executing any kernel:
                # drop every cached pack so the eager path rebuilds them
                self.G.invalidate()
                for sd in self.D.subs:
                    sd.invalidate()
            self.stamps.force = False
            graphs[key] = entry
        if entry == "eager":
            return self.step(x, y, y_mel)
        entry[5] += 1
        g, sx, sy, sm, out = entry[:5]
        sx.copy_(x); sy.copy_(y); sm.copy_(y_mel)
        g.replay()
        return out

    # Data-parallel: the all-reduces of one NCCL communicator execute one at a time in issue order, so a gradient
    # slice queued behind the slice of a lane whose backward ends later waits for that lane (measured at 2 GPUs,
    # profiles/r02_summary.md section 5: the second scale discriminator ended its backward at 3.6 ms and got its
    # slice back at 8.8 ms, behind the spectral-norm scale's).  The first data-parallel captures therefore carry
    # hg_timestamp marks: after CALIBRATION_REPLAYS replays the lanes are re-sorted by the time their backward
    # ended and the step is captured again — up to CALIBRATION_ROUNDS times, because the new order moves the lanes'
    # timings — and the order with the earliest end of step is captured for good, without marks.  Rank 0 decides
    # and broadcasts: every rank must issue the same order.
    CALIBRATION_REPLAYS = 3
    CALIBRATION_ROUNDS = 3

    @property
    def warmup_calls(self) -> int:
        """step_graphed calls before the final graph replays: eager, capture, (data-parallel: calibration rounds)"""
        if self.world == 1 or self.D.order_fixed:
            return 2
        return 2 + self.CALIBRATION_ROUNDS * (self.CALIBRATION_REPLAYS + 1)

    def _calibrate_slice_order(self) -> None:
        torch.cuda.synchronize()
        t = self.stamps.read()
        n = len(self.D.subs)
        cal = self.__dict__.setdefault("_cal", {"tried": [], "best": None})
        cur = list(self.D.order)
        cal["tried"].append(cur)
        end = t.get("end", float("inf"))
        if cal["best"] is None or end < cal["best"][0]:
            cal["best"] = (end, cur)
        nxt = sorted(range(n), key=lambda i: t.get(f"d{i}_bwd_done", float(i)))
        final = len(cal["tried"]) >= self.CALIBRATION_ROUNDS or nxt in cal["tried"]
        msg = torch.tensor([int(final)] + (cal["best"][1] if final else nxt), dtype=torch.int64, device=self.device)
        src = 0 if self.pg is None else torch.distributed.get_global_rank(self.pg, 0)
        torch.distributed.broadcast(msg, src=src, group=self.pg)
        msg = [int(v) for v in msg.cpu().tolist()]
        self.D.order = msg[1:]
        self.D.order_fixed = bool(msg[0])
        self.slice_order_log = cal["tried"], cal["best"]
