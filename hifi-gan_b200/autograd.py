"""torch.autograd bindings of the backward kernels: the reference's modules are ordinary differentiable nn.Modules
(src/models.py:100-116, 142-161, 206-216; src/meldataset.py:56-85), and an UPSTREAM-style loop does

    loss.backward(); optim.step()          # torch.optim.AdamW over generator.parameters() / chain(msd, mpd)

through them (SURVEY.md §3.3).  This module makes `Generator(x)`, `DiscriminatorP/S(x)` (hence `mpd(y, y_hat)`,
`msd(y, y_hat)`), `mel_spectrogram(y)` and the three loss functions work under that loop: each is ONE
`torch.autograd.Function` whose forward and backward are the library's kernels (the same ones `TrainStep` drives —
`GeneratorTrainer` / `_SubDiscTrainer` in train.py own the chain rule).  `TrainStep` remains the fast path (one CUDA
graph, fused optimizer, fused losses); this is the drop-in path.

Contract and limits (each raises loudly, there is no fallback to torch ops):
  * parameters must be contiguous fp32 CUDA tensors (what `module.cuda()` gives);
  * only the MOST RECENT forward of a Generator can be differentiated (its saved activations live in one workspace);
    a discriminator keeps its four most recent calls (the UPSTREAM step needs two per backward);
  * no double backward.
Numerics as everywhere else: bf16 operands / stored activations and activation gradients, fp32 accumulation, fp32
parameter gradients.
"""
from __future__ import annotations

import itertools
from typing import List, Optional

import torch

from . import _lib
from .models import _avgpool, _loss_mean, _stream


def _engine(module: torch.nn.Module, device, build):
    """The module's autograd-path engine (`build()` makes one).  Its job tables hold raw pointers to the parameters
    and buffers, so it is rebuilt whenever their storage moved: `.to()`, `p.data = ...`, FlatParams re-pointing them."""
    key = (device,) + tuple(t.data_ptr() for t in itertools.chain(module.parameters(), module.buffers()))
    eng = module.__dict__.get("_hg_autograd")
    if eng is None or eng.storage_key != key:
        eng = build()
        eng.storage_key = key
        module.__dict__["_hg_autograd"] = eng
    return eng


def _grads_out(flat, params, needs) -> list:
    """copies of the private flat gradient buffer, one view per parameter that wants a gradient (torch may keep the
    returned tensors as `.grad`, and the buffer is rewritten by the next backward)"""
    snap = flat.g.clone()
    return [snap[o:o + n].view(p.shape) if need else None
            for p, o, n, need in zip(params, flat.offsets, flat.sizes, needs)]


# ---------------------------------------------------------------------------------------------------- Generator
class _GeneratorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gen, *params):
        from .train import GeneratorTrainer
        tr = _engine(gen, x.device, lambda: GeneratorTrainer(gen, x.device, bind=False))
        y = tr.forward(x.detach())
        tr.call_id = getattr(tr, "call_id", 0) + 1
        ctx.tr, ctx.call_id, ctx.in_shape = tr, tr.call_id, tuple(x.shape)
        ctx.set_materialize_grads(False)
        return y.clone()

    @staticmethod
    def backward(ctx, dy):
        tr = ctx.tr
        if dy is None:
            return (None, None) + (None,) * len(tr.flat.params)
        if tr.call_id != ctx.call_id:
            raise RuntimeError("hifigan_b200: only the most recent Generator forward can be differentiated "
                               "(its saved activations were overwritten by a later call)")
        dx = None
        if ctx.needs_input_grad[0]:
            b, c, f = ctx.in_shape
            dx_p = torch.empty(b, tr.eng.pre.cin_p, f, dtype=torch.float32, device=dy.device)
        else:
            dx_p = None
        tr.backward(dy.contiguous().float(), dx_mel=dx_p)
        if dx_p is not None:
            dx = dx_p[:, : ctx.in_shape[1]].contiguous()
        return (dx, None) + tuple(_grads_out(tr.flat, tr.flat.params, ctx.needs_input_grad[2:]))


def generator_forward(gen, x: torch.Tensor) -> torch.Tensor:
    return _GeneratorFn.apply(x, gen, *gen.parameters())


# ----------------------------------------------------------------------------------------------- discriminators
_SLOTS = 4


class _DiscEngine:
    """Per-module state of a DiscriminatorP / DiscriminatorS: the sub-discriminator trainer (kernel sequences,
    workspaces), a private flat gradient buffer and the ring of call slots."""

    def __init__(self, disc, device):
        from .train import FlatParams, _SubDiscTrainer
        self.flat = FlatParams(disc, device, bind=False)
        self.sd = _SubDiscTrainer(disc, device, self.flat, nslots=_SLOTS)
        self.next_slot = 0
        self.slot_call = [0] * _SLOTS
        self.calls = 0


def _disc_run(disc, x: torch.Tensor, differentiable: bool):
    """One call of a sub-discriminator: claim the next ring slot, run the forward, export the feature maps and
    assemble the logits.  Returns (feature maps fp32 [B,C,H,p] + logits [B,1,H,p],
    (engine, slot, call id, G, the slot's weights and banks, x2d))."""
    eng = _engine(disc, x.device, lambda: _DiscEngine(disc, x.device))
    sd = eng.sd
    L = _lib.lib()
    b, c, t = x.shape
    if c != 1:
        raise ValueError("discriminators take [B,1,T] audio")
    x2d = x.detach().reshape(b, t).contiguous().float()
    slot = eng.next_slot
    eng.next_slot = (slot + 1) % _SLOTS
    eng.calls += 1
    eng.slot_call[slot] = eng.calls
    G, cs = sd.forward_single(x2d, slot, dgrad=differentiable)
    period, st = sd.period, _stream()
    outs = []
    for (h, rows, ch), act in zip(G["geo"], G["act"]):
        f = torch.empty(b, ch, h, period, dtype=torch.float32, device=x.device)
        _lib.check(L.hg_disc_export_fmap(act.data_ptr(), b, period, h, rows, ch, f.data_ptr(), st),
                   "hg_disc_export_fmap")
        outs.append(f)
    h_last = G["geo"][-1][0]
    post = G["logit"].view(b, period, h_last).permute(0, 2, 1).contiguous().unsqueeze(1)     # [B,1,H,p]
    outs.append(post)
    return tuple(outs), (eng, slot, eng.calls, G, cs, x2d)


class _DiscFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, disc, *params):
        outs, (ctx.eng, ctx.slot, ctx.call, ctx.G, ctx.cs, ctx.x2d) = _disc_run(disc, x, True)
        ctx.set_materialize_grads(False)
        return outs

    @staticmethod
    def backward(ctx, *douts):
        eng, G = ctx.eng, ctx.G
        sd = eng.sd
        n_par = len(eng.flat.params)
        if all(d is None for d in douts):
            return (None, None) + (None,) * n_par
        if eng.slot_call[ctx.slot] != ctx.call:
            raise RuntimeError(f"hifigan_b200: a discriminator keeps the activations of its {_SLOTS} most recent calls; "
                               "this call's were overwritten before backward")
        L = _lib.lib()
        st = _stream()
        b, t = ctx.x2d.shape
        period = sd.period
        nl = len(sd.mids)
        pre: List[Optional[torch.Tensor]] = []
        for l, ((h, rows, ch), d) in enumerate(zip(G["geo"], douts[: nl + 1])):
            if d is None:
                pre.append(None)
                continue
            buf = G.setdefault("pre", {}).get(l)
            if buf is None:
                buf = G["pre"][l] = torch.zeros_like(G["act"][l])
            _lib.check(L.hg_disc_import_fmap(d.contiguous().float().data_ptr(), b, period, h, rows, ch, buf.data_ptr(),
                                             st), "hg_disc_import_fmap")
            pre.append(buf)
        h_last = G["geo"][-1][0]
        dpost = douts[nl + 1]
        if dpost is None:
            dlogit = torch.zeros(b * period, h_last, dtype=torch.float32, device=ctx.x2d.device)
        else:                                               # [B,1,H,p] -> the internal [B*p][H]
            dlogit = dpost.float().reshape(b, h_last, period).permute(0, 2, 1).reshape(b * period, h_last).contiguous()
        want_w = any(ctx.needs_input_grad[2:])
        dy = torch.zeros(b, t, dtype=torch.float32, device=ctx.x2d.device) if ctx.needs_input_grad[0] else None
        if want_w:
            eng.flat.g.zero_()
        sd.backward_single(G, ctx.cs, ctx.x2d, dlogit, pre, want_w, dy)
        grads = _grads_out(eng.flat, eng.flat.params, ctx.needs_input_grad[2:]) if want_w else [None] * n_par
        return (None if dy is None else dy.view(b, 1, t), None) + tuple(grads)


def disc_forward(disc, x: torch.Tensor, differentiable: bool):
    """(flattened logits, feature maps fp32 [B,C,H,p]) of one DiscriminatorP / DiscriminatorS call; through autograd
    when `differentiable`, otherwise the same forward without the data-gradient banks"""
    outs = _DiscFn.apply(x, disc, *disc.parameters()) if differentiable else _disc_run(disc, x, False)[0]
    fmap = list(outs)
    return torch.flatten(fmap[-1], 1, -1), fmap


class _AvgPoolFn(torch.autograd.Function):
    """AvgPool1d(4, 2, padding=2) (src/models.py:227-230) on hg_avgpool_4_2_2_fwd / _bwd"""

    @staticmethod
    def forward(ctx, x):
        ctx.shape = tuple(x.shape)
        return _avgpool(x)

    @staticmethod
    def backward(ctx, dout):
        b, c, t = ctx.shape
        din = torch.zeros(b * c, t, dtype=torch.float32, device=dout.device)
        d = dout.reshape(b * c, -1).contiguous().float()
        _lib.check(_lib.lib().hg_avgpool_4_2_2_bwd(d.data_ptr(), b * c, t, din.data_ptr(), _stream()),
                   "hg_avgpool_4_2_2_bwd")
        return din.view(b, c, t)


def avgpool(x: torch.Tensor) -> torch.Tensor:
    return _AvgPoolFn.apply(x)


# ------------------------------------------------------------------------------------------------------ losses
class _MeanFn(torch.autograd.Function):
    """mode 0: mean |a - b|;  mode 1: mean (c - a)^2   (hg_loss_sum forward, hg_loss_grad backward)"""

    @staticmethod
    def forward(ctx, a, b, mode, c):
        a32 = a.detach().contiguous().float()
        b32 = None if b is None else b.detach().contiguous().float()
        ctx.a, ctx.b, ctx.mode, ctx.c = a32, b32, mode, c
        ctx.a_shape, ctx.b_shape = a.shape, (None if b is None else b.shape)
        return _loss_mean(a32, b32, mode, c)

    @staticmethod
    def backward(ctx, dout):
        a, b, mode, c = ctx.a, ctx.b, ctx.mode, ctx.c
        n = a.numel()
        L = _lib.lib()
        st = _stream()
        ga = gb = None
        # d mean|a-b| / da = sgn(a-b) / n;  d mean (c-a)^2 / da = 2 (a-c) / n;  then times the incoming scalar
        sc = dout.detach().reshape(1).float().contiguous()       # the incoming scalar stays on the device
        if ctx.needs_input_grad[0]:
            ga = torch.empty_like(a)
            if mode == 0:
                _lib.check(L.hg_loss_grad(a.data_ptr(), b.data_ptr(), n, 0, 0.0, 1.0 / n, 0.0, sc.data_ptr(),
                                          ga.data_ptr(), st), "hg_loss_grad")
            else:
                _lib.check(L.hg_loss_grad(a.data_ptr(), 0, n, 1, c, 2.0 / n, 0.0, sc.data_ptr(), ga.data_ptr(), st),
                           "hg_loss_grad")
            ga = ga.view(ctx.a_shape)
        if b is not None and ctx.needs_input_grad[1]:
            gb = torch.empty_like(b)
            _lib.check(L.hg_loss_grad(b.data_ptr(), a.data_ptr(), n, 0, 0.0, 1.0 / n, 0.0, sc.data_ptr(), gb.data_ptr(),
                                      st), "hg_loss_grad")
            gb = gb.view(ctx.b_shape)
        return ga, gb, None, None


def device_mean(a: torch.Tensor, b: Optional[torch.Tensor], mode: int, c: float) -> torch.Tensor:
    if not a.is_cuda or (b is not None and not b.is_cuda):
        raise RuntimeError("hifigan_b200 losses have no CPU path; move the tensors to a B200")
    return _MeanFn.apply(a, b, mode, c)


# --------------------------------------------------------------------------------------------------------- mel
class _MelFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y2, plan, minmax_ptr):
        b, t = y2.shape
        yin = y2.detach()
        out = torch.empty(b, plan.num_mels, plan.frames(t), dtype=torch.float32, device=y2.device)
        _lib.check(_lib.lib().hg_mel_fwd(plan.handle, yin.data_ptr(), b, t, out.data_ptr(), minmax_ptr, _stream()),
                   "hg_mel_fwd")
        ctx.plan, ctx.y = plan, yin
        return out

    @staticmethod
    def backward(ctx, dmel):
        if dmel is None:
            return None, None, None
        y = ctx.y
        b, t = y.shape
        dy = torch.zeros_like(y)
        dm = dmel.contiguous().float()
        _lib.check(_lib.lib().hg_mel_bwd(ctx.plan.handle, y.data_ptr(), dm.data_ptr(), b, t, dy.data_ptr(), _stream()),
                   "hg_mel_bwd")
        return dy, None, None


def mel_forward(y2: torch.Tensor, plan, minmax_ptr: int) -> torch.Tensor:
    """y2 fp32 contiguous [B, T] -> log-mel [B, num_mels, frames], differentiable w.r.t. y2 (hg_mel_bwd)"""
    return _MelFn.apply(y2, plan, minmax_ptr)
