"""HiFi-GAN vocoder models on hand-written sm_100a kernels — drop-in for the reference's src/models.py.

Same public names, constructor arguments, attribute names and state_dict keys as the reference
(`Generator` models.py:75-125, `ResBlock1` :11-48, `ResBlock2` :51-72, the discriminators :128-248 and the
three losses :251-282), so existing configs and checkpoints load unchanged.  The torch modules held by
these classes are *parameter containers only*: their `forward` is never called.  All arithmetic of
`Generator.forward` runs in libhifigan_b200.so (include/hifigan_b200.h):

    mel fp32 [B,80,F] --hg_ncl_to_nlc--> bf16 [B,F,128]
      --hg_conv1d_fwd (conv_pre, epilogue: bias + leaky_relu 0.1)-->
      per stage: hg_conv1d_fwd on polyphase-packed ConvTranspose1d weights  (raw + leaky_relu'd outputs)
                 3 MRF branches x (conv, conv) x 3 via hg_conv1d_fwd; residual add, branch average and the
                 next leaky_relu are fused into the last conv's epilogue
      --hg_conv_post_tanh_fwd--> fp32 [B,1,T]

Numerics (declared): bf16 operands and bf16-stored activations, fp32 accumulation and epilogue math.
There is no CPU path and no fallback: CPU tensors raise.
"""
from __future__ import annotations

import os
import warnings
from ctypes import byref, c_int
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn
from torch.nn import AvgPool1d, Conv1d, Conv2d, ConvTranspose1d
from torch.nn.utils import remove_weight_norm, spectral_norm, weight_norm

from . import _lib
from .utils import get_padding, init_weights

LRELU_SLOPE = 0.1


def _wn(module: nn.Module) -> nn.Module:
    """Old-style weight_norm (keys weight_g / weight_v) — the checkpoint contract (SURVEY.md §8b)."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return weight_norm(module)


def _pad_ch(c: int) -> int:
    """Channel count as laid out in HBM: 32, or a multiple of 64 (one 128-byte swizzle row per 64)."""
    return 32 if c <= 32 else (c + 63) // 64 * 64


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(x: torch.Tensor, what: str) -> None:
    if not x.is_cuda:
        raise RuntimeError(f"{what}: hifigan_b200 has no CPU path; move the tensor to a B200 (got {x.device})")


def _wants_grad(x: torch.Tensor, module: nn.Module) -> bool:
    """whether torch autograd records this call of `module` on `x`"""
    return torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in module.parameters()))


def _g_v(m: nn.Module) -> Tuple[Optional[torch.Tensor], torch.Tensor]:
    """(g, v) while weight_norm is attached, (None, weight) after remove_weight_norm."""
    if hasattr(m, "weight_g"):
        return m.weight_g, m.weight_v
    return None, m.weight


class _PackedConv:
    """One conv layer in GEMM-ready form: bf16 [taps][cout_p][cin_p] + fp32 bias [cout_p]."""

    __slots__ = ("module", "kind", "cin", "cout", "cin_p", "cout_p", "taps", "dil", "pad_left", "stride",
                 "w", "bias", "key")

    def __init__(self, module: nn.Module, kind: str, device):
        self.module, self.kind = module, kind
        g, v = _g_v(module)
        if kind == "conv":
            cout, cin, k = v.shape
            self.cin, self.cout, self.taps = cin, cout, k
            self.dil = module.dilation[0]
            self.pad_left = module.padding[0]
            self.stride = 1
            self.cin_p, self.cout_p = _pad_ch(cin), _pad_ch(cout)
            n_rows = self.cout_p
        else:  # ConvTranspose1d -> polyphase 1-D conv producing [T_in][stride*cout_p]
            cin, cout, k = v.shape
            u, pad = module.stride[0], module.padding[0]
            nshift, smin = c_int(), c_int()
            _lib.check(_lib.lib().hg_convtr1d_geometry(k, u, pad, byref(nshift), byref(smin)))
            if k - 2 * pad != u or module.output_padding[0] != 0:
                raise NotImplementedError("ConvTranspose1d must satisfy out_len == stride * in_len")
            self.cin, self.cout, self.taps = cin, cout, nshift.value
            self.dil, self.pad_left, self.stride = 1, -smin.value, u
            self.cin_p, self.cout_p = _pad_ch(cin), _pad_ch(cout)
            n_rows = u * self.cout_p
        self.w = torch.empty(self.taps, n_rows, self.cin_p, dtype=torch.bfloat16, device=device)
        self.bias = torch.zeros(n_rows, dtype=torch.float32, device=device)
        self.key = None

    def _fingerprint(self):
        g, v = _g_v(self.module)
        b = self.module.bias
        return tuple((t.data_ptr(), t._version) for t in (g, v, b) if t is not None)

    def tensors(self):
        g, v = _g_v(self.module)
        return [t for t in (g, v, self.module.bias) if t is not None]

    def batchable(self) -> bool:
        """parameters the batched pack kernel can read in place: contiguous fp32 on the pack's device"""
        return all(t.device == self.w.device and t.dtype == torch.float32 and t.is_contiguous() for t in self.tensors())

    def add_pack_job(self, table, phase: str) -> None:
        """this layer's fold + pack as one job of a batched launch (batched.py / hg_prep_batched)"""
        from . import batched
        m = self.module
        g, v = _g_v(m)
        if self.bias.data_ptr() in [t.data_ptr() for t in self.tensors()]:     # refresh() may have aliased the parameter
            self.bias = torch.zeros(self.w.shape[1], dtype=torch.float32, device=self.w.device)
        if self.kind == "conv":
            table.add(phase, batched.GEN_CONV, self.cout_p, 0, v, g, m.bias, self.w, self.bias,
                      ints=(self.cout, self.cin, self.taps, self.cout_p, self.cin_p))
        else:
            nshift, smin = c_int(), c_int()
            _lib.check(_lib.lib().hg_convtr1d_geometry(m.kernel_size[0], self.stride, m.padding[0], byref(nshift),
                                                       byref(smin)))
            table.add(phase, batched.GEN_CONVTR, self.cin_p, 0, v, g, m.bias, self.w, self.bias,
                      ints=(self.cin, self.cout, m.kernel_size[0], self.cin_p, self.cout_p, self.stride, m.padding[0],
                            nshift.value, smin.value))

    def refresh(self) -> None:
        """(Re)pack when a parameter changed: weight_norm fold + bf16 GEMM layout (hg_pack_*)."""
        key = self._fingerprint()
        # (data_ptr, _version) cannot see writes through raw pointers (the AdamW kernel), and a captured graph must
        # hold the re-pack launches whatever the host cache says: never skip while a stream is capturing
        if key == self.key and not torch.cuda.is_current_stream_capturing():
            return
        L = _lib.lib()
        m = self.module
        g, v = _g_v(m)
        dev = self.w.device
        v = v.detach().to(device=dev, dtype=torch.float32)
        g = None if g is None else g.detach().to(device=dev, dtype=torch.float32).reshape(-1)
        b = m.bias.detach().to(device=dev, dtype=torch.float32) if m.bias is not None else None
        if self.kind == "conv":
            if self.cout_p != self.cout:  # zero rows for padded output channels
                v = torch.cat([v, v.new_zeros(self.cout_p - self.cout, *v.shape[1:])], 0)
                if g is not None:
                    g = torch.cat([g, g.new_zeros(self.cout_p - self.cout)], 0)
            v = v.contiguous()
            _lib.check(L.hg_pack_conv1d_weight(v.data_ptr(), 0 if g is None else g.contiguous().data_ptr(),
                                               self.cout_p, self.cin, self.taps, self.cin_p,
                                               self.w.data_ptr(), _stream()), "hg_pack_conv1d_weight")
            if b is not None and self.cout_p == self.cout and b.is_contiguous():
                self.bias = b           # no padding: read the parameter in place (no copy kernel per step)
            else:
                self.bias.zero_()
                if b is not None:
                    self.bias[: self.cout].copy_(b)
        else:
            k = m.kernel_size[0]
            if self.cout_p != self.cout or self.cin_p != self.cin:
                vp = v.new_zeros(self.cin_p, self.cout_p, k)
                vp[: self.cin, : self.cout] = v
                v = vp
                if g is not None:
                    g = torch.cat([g, g.new_zeros(self.cin_p - self.cin)], 0)
            v = v.contiguous()
            _lib.check(L.hg_pack_convtr1d_weight(v.data_ptr(), 0 if g is None else g.contiguous().data_ptr(),
                                                 self.cin_p, self.cout_p, k, self.stride, m.padding[0],
                                                 self.w.data_ptr(), _stream()), "hg_pack_convtr1d_weight")
            self.bias.zero_()
            if b is not None:
                self.bias.view(self.stride, self.cout_p)[:, : self.cout].copy_(b.unsqueeze(0).expand(self.stride, -1))
        self.key = key


def _conv(L, x, pc: _PackedConv, batch: int, t: int, *, res=(None, None, None), res0_slope=0.0, scale=1.0,
          out_raw=None, out_act=None, slope=LRELU_SLOPE, item=(0, 1)) -> None:
    """item = (device pointer of int32 item lengths or 0, rows per length unit): ragged batches, see hg_conv1d_fwd.
    res0_slope > 0: res[0] holds leaky_relu(residual, res0_slope), undone in the epilogue (hg_conv1d_fwd_actres)."""
    p = [0 if r is None else r.data_ptr() for r in res]
    outs = (0 if out_raw is None else out_raw.data_ptr(), 0 if out_act is None else out_act.data_ptr(), slope,
            item[0], item[1], _stream())
    head = (x.data_ptr(), pc.w.data_ptr(), pc.bias.data_ptr(), batch, t, pc.cin_p, pc.w.shape[1], pc.taps, pc.dil,
            pc.pad_left)
    if res0_slope:
        _lib.check(L.hg_conv1d_fwd_actres(*head, p[0], res0_slope, p[1], p[2], scale, *outs), "hg_conv1d_fwd_actres")
    else:
        _lib.check(L.hg_conv1d_fwd(*head, p[0], p[1], p[2], scale, *outs), "hg_conv1d_fwd")


def _pair(L, x, pc1: _PackedConv, pc2: _PackedConv, batch: int, t: int, *, x_act=False, res=(None, None),
          scale=1.0, out_raw=None, out_act=None, slope=LRELU_SLOPE, item=(0, 1)) -> None:
    """One fused ResBlock1 step: conv2(lrelu(conv1(lrelu(x)) + b1)) + b2 + x (+ res) — hg_resblock_pair_fwd.
    x_act: x holds leaky_relu(x, LRELU_SLOPE) (hg_resblock_pair_fwd_actin)."""
    p = [0 if r is None else r.data_ptr() for r in res]
    w2, b2 = (0, 0) if pc2 is None else (pc2.w.data_ptr(), pc2.bias.data_ptr())   # None: one ResBlock2 step
    fn, name = ((L.hg_resblock_pair_fwd_actin, "hg_resblock_pair_fwd_actin") if x_act
                else (L.hg_resblock_pair_fwd, "hg_resblock_pair_fwd"))
    _lib.check(fn(x.data_ptr(), pc1.w.data_ptr(), pc1.bias.data_ptr(), w2, b2, batch, t, pc1.cin_p, pc1.taps,
                  pc1.dil, LRELU_SLOPE, p[0], p[1], scale, 0 if out_raw is None else out_raw.data_ptr(),
                  0 if out_act is None else out_act.data_ptr(), slope, item[0], item[1], _stream()), name)


_FUSE_PAIRS = True  # tests flip this to compare the fused and the two-launch paths


def _pair_ok(L, pc1: _PackedConv, pc2: _PackedConv) -> bool:
    return bool(_FUSE_PAIRS and pc1.cin_p == pc1.cout_p == pc2.cin_p == pc2.cout_p and pc1.taps == pc2.taps
                and pc2.dil == 1 and L.hg_resblock_pair_supported(pc1.cin_p, pc1.taps, pc1.dil))


def _single_ok(L, pc: _PackedConv) -> bool:
    return bool(_FUSE_PAIRS and pc.cin_p == pc.cout_p and L.hg_resblock_single_supported(pc.cin_p, pc.taps, pc.dil))


def _block_plan(L, block: "nn.Module", packs: List[_PackedConv]) -> List[bool]:
    """Per ResBlock step: True when it runs as ONE fused launch (conv-lrelu-conv-residual for ResBlock1,
    lrelu-conv-residual for ResBlock2)."""
    if not isinstance(block, ResBlock1):
        return [_single_ok(L, pc) for pc in packs]
    return [_pair_ok(L, packs[2 * i], packs[2 * i + 1]) for i in range(len(packs) // 2)]


def _resblock_chain(L, block: "nn.Module", packs: List[_PackedConv], batch: int, t: int, c_p: int,
                    x_raw, x_act, bufs: Dict[str, torch.Tensor], final, item=(0, 1)) -> None:
    """Run one ResBlock (type 1: packs = [c1_0, c2_0, c1_1, ...]; type 2: packs = [c_0, c_1, ...]).
    `final(kw)` issues the LAST launch of the block (so the caller can fuse the MRF average): kw is either
    dict(pair=(pc1, pc2), x=input, x_act=bool) or dict(pc=conv, x=activated_input, res0=residual, res0_slope=s).
    A step's input is stored once: raw when the step is fused (the pair kernel applies the leaky_relu itself),
    leaky_relu'd when it is not (its convs read that copy and the residual add undoes the activation, res0_slope).
    x_raw or x_act may be None; a fused step reads x_raw when it exists."""
    two_conv = isinstance(block, ResBlock1)
    fused = _block_plan(L, block, packs)
    steps = len(fused)
    cur_raw, cur_act = x_raw, x_act
    ping = [(bufs["a_raw"], bufs["a_act"]), (bufs["b_raw"], bufs["b_act"])]
    for i in range(steps):
        last = i == steps - 1
        nr, na = ping[i & 1]
        if not last:   # the one copy the next step reads
            nr, na = (nr, None) if fused[i + 1] else (None, na)
        if fused[i]:
            pc1, pc2 = (packs[2 * i], packs[2 * i + 1]) if two_conv else (packs[i], None)
            x, x_is_act = (cur_raw, False) if cur_raw is not None else (cur_act, True)
            if last:
                final(dict(pair=(pc1, pc2), x=x, x_act=x_is_act))
            else:
                _pair(L, x, pc1, pc2, batch, t, x_act=x_is_act, out_raw=nr, out_act=na, item=item)
        else:
            if two_conv:
                _conv(L, cur_act, packs[2 * i], batch, t, out_act=bufs["t1"], item=item)
                src, pc = bufs["t1"], packs[2 * i + 1]
            else:
                src, pc = cur_act, packs[i]
            res0, res0_slope = (cur_raw, 0.0) if cur_raw is not None else (cur_act, LRELU_SLOPE)
            if last:
                final(dict(pc=pc, x=src, res0=res0, res0_slope=res0_slope))
            else:
                _conv(L, src, pc, batch, t, res=(res0, None, None), res0_slope=res0_slope, out_raw=nr, out_act=na,
                      item=item)
        cur_raw, cur_act = nr, na


class _StandaloneBlockMixin:
    """forward() for a ResBlock used on its own (x fp32 [B,C,T] -> fp32 [B,C,T]) on the same kernels."""

    def _packs(self, device) -> List[_PackedConv]:
        cache = self.__dict__.setdefault("_hg_packs", None)
        convs = self._ordered_convs()
        if cache is None or cache[0].w.device != device:
            cache = [_PackedConv(m, "conv", device) for m in convs]
            self.__dict__["_hg_packs"] = cache
        for pc in cache:
            pc.refresh()
        return cache

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        _require_cuda(x, type(self).__name__)
        if _wants_grad(x, self):
            raise NotImplementedError(f"{type(self).__name__} on its own is an inference surface (call it under "
                                      "torch.no_grad()); it is differentiable as part of Generator")
        L = _lib.lib()
        b, c, t = x.shape
        packs = self._packs(x.device)
        c_p = packs[0].cin_p
        mk = lambda: torch.empty(b, t, c_p, dtype=torch.bfloat16, device=x.device)
        bufs = {k: mk() for k in ("x_raw", "x_act", "t1", "a_raw", "a_act", "b_raw", "b_act", "out")}
        xin = x.contiguous().float()
        _lib.check(L.hg_ncl_to_nlc(xin.data_ptr(), b, c, t, c_p, bufs["x_raw"].data_ptr(),
                                   bufs["x_act"].data_ptr(), LRELU_SLOPE, _stream()), "hg_ncl_to_nlc")

        def final(kw):
            if "pair" in kw:
                _pair(L, kw["x"], *kw["pair"], b, t, x_act=kw["x_act"], out_raw=bufs["out"])
            else:
                _conv(L, kw["x"], kw["pc"], b, t, res=(kw["res0"], None, None), res0_slope=kw["res0_slope"],
                      out_raw=bufs["out"])

        _resblock_chain(L, self, packs, b, t, c_p, bufs["x_raw"], bufs["x_act"], bufs, final)
        y = torch.empty(b, c_p, t, dtype=torch.float32, device=x.device)
        _lib.check(L.hg_nlc_to_ncl(bufs["out"].data_ptr(), b, t, c_p, y.data_ptr(), _stream()), "hg_nlc_to_ncl")
        return y[:, :c].contiguous() if c_p != c else y


class ResBlock1(_StandaloneBlockMixin, torch.nn.Module):
    """3 x (lrelu -> dilated conv -> lrelu -> conv -> + x); reference src/models.py:11-48."""

    def __init__(self, h, channels, kernel_size=3, dilation=(1, 3, 5)):
        super().__init__()
        self.h = h

        def conv(d):
            return _wn(Conv1d(channels, channels, kernel_size, 1, dilation=d,
                              padding=get_padding(kernel_size, d)))

        # creation / init order fixes the RNG stream; it is part of same-seed parity (SURVEY App. B.4)
        self.convs1 = nn.ModuleList([conv(d) for d in dilation[:3]])
        self.convs1.apply(init_weights)
        self.convs2 = nn.ModuleList([conv(1) for _ in dilation[:3]])
        self.convs2.apply(init_weights)

    def _ordered_convs(self):
        out = []
        for c1, c2 in zip(self.convs1, self.convs2):
            out += [c1, c2]
        return out

    def remove_weight_norm(self):
        for m in list(self.convs1) + list(self.convs2):
            remove_weight_norm(m)


class ResBlock2(_StandaloneBlockMixin, torch.nn.Module):
    """2 x (lrelu -> dilated conv -> + x); reference src/models.py:51-72."""

    def __init__(self, h, channels, kernel_size=3, dilation=(1, 3)):
        super().__init__()
        self.h = h
        self.convs = nn.ModuleList([
            _wn(Conv1d(channels, channels, kernel_size, 1, dilation=d, padding=get_padding(kernel_size, d)))
            for d in dilation[:2]])
        self.convs.apply(init_weights)

    def _ordered_convs(self):
        return list(self.convs)

    def remove_weight_norm(self):
        for m in self.convs:
            remove_weight_norm(m)


class _GeneratorEngine:
    """Packed weights, workspaces and the kernel sequence of one Generator on one device."""

    def __init__(self, gen: "Generator", device):
        self.gen, self.device = gen, device
        self.pre = _PackedConv(gen.conv_pre, "conv", device)
        self.ups = [_PackedConv(m, "convtr", device) for m in gen.ups]
        self.blocks = [[_PackedConv(m, "conv", device) for m in rb._ordered_convs()] for rb in gen.resblocks]
        post = gen.conv_post
        self.post_cin_p = _pad_ch(post.in_channels)
        self.post_w = torch.zeros(self.post_cin_p, post.kernel_size[0], dtype=torch.float32, device=device)
        self.post_b = torch.zeros(1, dtype=torch.float32, device=device)
        self.post_key = None
        self.table, self.table_ptrs, self.ver_key = None, None, None
        self.ws: Dict[Tuple[int, int], Dict[str, torch.Tensor]] = {}
        self.graphs: Dict[tuple, tuple] = {}
        self.graph_seen = set()

    def packs(self) -> List[_PackedConv]:
        return [self.pre] + self.ups + [pc for blk in self.blocks for pc in blk]

    def _post_tensors(self):
        post = self.gen.conv_post
        g, v = _g_v(post)
        return [t for t in (g, v, post.bias) if t is not None]

    def refresh(self) -> None:
        """(Re)derive every filter bank from the parameters when any of them changed: weight_norm fold + bf16 GEMM
        layout for all layers in ONE launch (hg_prep_batched over a device-resident job table)."""
        packs = self.packs()
        tensors = [t for pc in packs for t in pc.tensors()] + self._post_tensors()
        if not all(pc.batchable() for pc in packs) or not all(
                t.device == self.post_w.device and t.dtype == torch.float32 and t.is_contiguous() for t in self._post_tensors()):
            return self._refresh_per_layer()            # parameters living elsewhere (a CPU module): staged per layer
        ptr_key = tuple(t.data_ptr() for t in tensors)
        ver_key = tuple(t._version for t in tensors)
        if self.table is None or ptr_key != self.table_ptrs:
            from . import batched
            table = batched.JobTable(self.device)
            for pc in packs:
                pc.add_pack_job(table, "pack")
            post = self.gen.conv_post
            g, v = _g_v(post)
            table.add("pack", batched.GEN_POST, 1, 0, v, g, post.bias, self.post_w, self.post_b,
                      ints=(post.in_channels, post.kernel_size[0], self.post_cin_p))
            self.table, self.table_ptrs, self.ver_key = table.finalize(), ptr_key, None
        # (data_ptr, _version) cannot see writes through raw pointers (the AdamW kernel: invalidate() clears the key),
        # and a captured graph must hold the re-pack launch whatever the host cache says
        if ver_key != self.ver_key or torch.cuda.is_current_stream_capturing():
            self.table.launch("pack")
            self.ver_key = ver_key

    def invalidate(self) -> None:
        self.ver_key = None
        self.post_key = None
        for pc in self.packs():
            pc.key = None

    def _refresh_per_layer(self) -> None:
        self.pre.refresh()
        for pc in self.ups:
            pc.refresh()
        for blk in self.blocks:
            for pc in blk:
                pc.refresh()
        post = self.gen.conv_post
        g, v = _g_v(post)
        key = tuple((t.data_ptr(), t._version) for t in (g, v, post.bias) if t is not None)
        if key != self.post_key or torch.cuda.is_current_stream_capturing():
            # single output channel, parameters not on this device: fold with torch on the way over
            v32 = v.detach().to(self.device, torch.float32)
            w = v32 if g is None else v32 * (g.detach().to(self.device, torch.float32)
                                             / v32.pow(2).sum(dim=(1, 2), keepdim=True).sqrt())
            self.post_w.zero_()
            self.post_w[: post.in_channels].copy_(w[0])
            self.post_b.copy_(post.bias.detach().to(self.device, torch.float32))
            self.post_key = key

    def workspace(self, batch: int, frames: int) -> Dict[str, torch.Tensor]:
        key = (batch, frames)
        ws = self.ws.get(key)
        if ws is not None:
            return ws
        gen = self.gen
        dev = self.device
        t, sizes = frames, []
        for pc in self.ups:
            t *= pc.stride
            sizes.append(batch * t * pc.cout_p)
        biggest = max(sizes)
        bf = lambda n: torch.empty(n, dtype=torch.bfloat16, device=dev)
        ws = {"mel": bf(batch * frames * self.pre.cin_p), "pre": bf(batch * frames * self.pre.cout_p)}
        names = ["x_raw", "x_act", "t1", "a_raw", "a_act", "b_raw", "b_act", "stage_out"]
        names += [f"r{j}" for j in range(max(1, gen.num_kernels - 1))]
        for n in names:
            ws[n] = bf(biggest)
        ws["y"] = torch.empty(batch, 1, t, dtype=torch.float32, device=dev)
        if len(self.ws) >= 8:  # bound the cache: workspaces for config 2 are ~10 GB
            old = next(iter(self.ws))
            self.ws.pop(old)
            for gk in [k for k in self.graphs if k[:2] == old]:
                self.graphs.pop(gk)      # a captured graph owns pointers into that workspace
        self.ws[key] = ws
        return ws

    # Small workloads are launch-bound (64 launches per V1 forward): replay them as one CUDA graph.
    GRAPH_MAX_SAMPLES = 1 << 21

    def forward(self, x: torch.Tensor, time_convs: bool = False, lengths: Optional[torch.Tensor] = None) -> torch.Tensor:
        """time_convs=True brackets the tensor-core conv launches (everything between the input transposition
        and conv_post) with CUDA events on the launching stream -> self.last_conv_events (bench.py roofline).
        lengths (int32 [B] on the device, frames per item): a ragged batch — see Generator.forward."""
        self.refresh()   # weight (re)packing stays outside any graph: it writes the same buffers in place
        b, c, frames = x.shape
        xin = x.contiguous()
        if xin.dtype != torch.float32:
            xin = xin.float()
        t_out = frames
        for pc in self.ups:
            t_out *= pc.stride
        use_graph = (not time_convs and lengths is None and b * t_out <= self.GRAPH_MAX_SAMPLES
                     and not os.environ.get("HG_DISABLE_GRAPHS") and not torch.cuda.is_current_stream_capturing())
        if not use_graph:
            return self._launch(xin, time_convs, lengths)
        key = (b, frames, _FUSE_PAIRS)
        entry = self.graphs.get(key)
        if entry is None:
            static_in = torch.empty_like(xin)
            static_in.copy_(xin)
            out = self._launch(static_in, False)    # eager run: one-time kernel loading / attribute setup, workspaces
            torch.cuda.synchronize()
            # capture on the SECOND call of a shape: the first call of a process can still be loading kernel
            # images lazily, which is not allowed while a stream is capturing
            if key not in self.graph_seen:
                self.graph_seen.add(key)
                return out
            try:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    out = self._launch(static_in, False)
                entry = (graph, static_in, out)
            except RuntimeError as e:               # stay correct: this shape keeps running eagerly
                warnings.warn(f"hifigan_b200: CUDA graph capture failed for shape {key}, running eagerly ({e})")
                torch.cuda.synchronize()
                entry = (None, None, None)
            if len(self.graphs) >= 8:
                self.graphs.pop(next(iter(self.graphs)))
            self.graphs[key] = entry
        graph, static_in, out = entry
        if graph is None:
            return self._launch(xin, False)
        static_in.copy_(xin)
        graph.replay()
        return out

    def _launch(self, xin: torch.Tensor, time_convs: bool, lengths: Optional[torch.Tensor] = None) -> torch.Tensor:
        L = _lib.lib()
        gen = self.gen
        b, c, frames = xin.shape
        ws = self.workspace(b, frames)
        nk = gen.num_kernels
        lp = 0 if lengths is None else lengths.data_ptr()     # ragged batch: per-item frame counts (device int32)
        mul = 1                                                # rows per frame at the current stage
        _lib.check(L.hg_ncl_to_nlc(xin.data_ptr(), b, c, frames, self.pre.cin_p, ws["mel"].data_ptr(), 0, 0.0,
                                   _stream()), "hg_ncl_to_nlc")
        if time_convs:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        # conv_pre; its only consumer is leaky_relu -> ups[0] (models.py:101-104)
        _conv(L, ws["mel"], self.pre, b, frames, out_act=ws["pre"], item=(lp, mul))
        cur, t = ws["pre"], frames
        for i, up in enumerate(self.ups):
            # The stage input is stored once: leaky_relu'd when a branch's first step is unfused (its convs read that
            # copy; the fused first steps of the other branches read it through hg_resblock_pair_fwd_actin), raw
            # when every first step is fused.
            need_act = any(not _block_plan(L, gen.resblocks[i * nk + j], self.blocks[i * nk + j])[0]
                           for j in range(nk))
            x_raw, x_act = (None, ws["x_act"]) if need_act else (ws["x_raw"], None)
            # polyphase: one output row of this launch is `stride` samples, so its valid rows are the INPUT's
            _conv(L, cur, up, b, t, out_raw=x_raw, out_act=x_act, item=(lp, mul))
            t *= up.stride
            mul *= up.stride
            c_p = up.cout_p
            last_stage = i == len(self.ups) - 1
            out_slope = 0.01 if last_stage else LRELU_SLOPE  # models.py:112 uses the default slope
            for j in range(nk):
                blk = gen.resblocks[i * nk + j]
                packs = self.blocks[i * nk + j]

                def final(kw, j=j):
                    if j < nk - 1:
                        # branch result; branches >= 2 of a wide MRF chain onto the running sum
                        others = (ws[f"r{j - 1}"] if (nk > 3 and j > 0) else None, None)
                        outs = dict(out_raw=ws[f"r{j}"])
                    else:
                        if nk > 3:
                            others = (ws[f"r{nk - 2}"], None)
                        else:
                            others = tuple(ws[f"r{q}"] for q in range(nk - 1)) + (None,) * (3 - nk)
                        outs = dict(scale=1.0 / nk, out_act=ws["stage_out"], slope=out_slope)
                    if "pair" in kw:
                        _pair(L, kw["x"], *kw["pair"], b, t, x_act=kw["x_act"], res=others, item=(lp, mul), **outs)
                    else:
                        _conv(L, kw["x"], kw["pc"], b, t, res=(kw["res0"],) + others, res0_slope=kw["res0_slope"],
                              item=(lp, mul), **outs)

                _resblock_chain(L, blk, packs, b, t, c_p, x_raw, x_act, ws, final, item=(lp, mul))
            cur = ws["stage_out"]
        if time_convs:
            ev1.record()
            self.last_conv_events = (ev0, ev1)
        post = gen.conv_post
        _lib.check(L.hg_conv_post_tanh_fwd(cur.data_ptr(), self.post_w.data_ptr(), self.post_b.data_ptr(), b, t,
                                           self.post_cin_p, post.kernel_size[0], ws["y"].data_ptr(), _stream()),
                   "hg_conv_post_tanh_fwd")
        return ws["y"]


class Generator(torch.nn.Module):
    """mel [B,80,F] -> waveform [B,1,F*prod(upsample_rates)]; reference src/models.py:75-125."""

    def __init__(self, h):
        super().__init__()
        self.h = h
        self.num_kernels = len(h.resblock_kernel_sizes)
        self.num_upsamples = len(h.upsample_rates)
        width = h.upsample_initial_channel
        self.conv_pre = _wn(Conv1d(80, width, 7, 1, padding=3))
        block_cls = ResBlock1 if h.resblock == '1' else ResBlock2  # string compare, as the reference

        self.ups = nn.ModuleList()
        for level, (rate, ksize) in enumerate(zip(h.upsample_rates, h.upsample_kernel_sizes)):
            self.ups.append(_wn(ConvTranspose1d(width >> level, width >> (level + 1), ksize, rate,
                                                padding=(ksize - rate) // 2)))
        self.resblocks = nn.ModuleList()
        for level in range(len(self.ups)):
            ch = width >> (level + 1)
            for ksize, dil in zip(h.resblock_kernel_sizes, h.resblock_dilation_sizes):
                self.resblocks.append(block_cls(h, ch, ksize, dil))
        self.conv_post = _wn(Conv1d(ch, 1, 7, 1, padding=3))
        self.ups.apply(init_weights)
        self.conv_post.apply(init_weights)
        self.__dict__["_hg_engines"] = {}

    def _engine(self, device) -> _GeneratorEngine:
        engines = self.__dict__.setdefault("_hg_engines", {})
        eng = engines.get(device)
        if eng is None:
            eng = _GeneratorEngine(self, device)
            engines[device] = eng
        return eng

    def forward(self, x: torch.Tensor, lengths: Optional[torch.Tensor] = None) -> torch.Tensor:
        """mel [B,80,F] -> waveform [B,1,T], a fresh tensor per call like the reference.  (`self._engine(dev)
        .forward(x)` returns the engine-owned buffer without the copy: the benchmark's device-resident path.)

        lengths (extension, inference only): int tensor [B] of frame counts for a RAGGED batch — item i is the mel
        x[i, :, :lengths[i]] (the rest of its row is ignored) and its waveform is out[i, 0, :lengths[i] * hop]; every
        layer treats the rows past an item's end as the zero padding the item would see if it ran alone, so the
        samples are bit-identical to the reference's one-utterance-per-call schedule (src/inference.py:55)."""
        _require_cuda(x, "Generator.forward")
        if x.dim() != 3 or x.shape[1] != self.conv_pre.in_channels:
            raise ValueError(f"expected [B,{self.conv_pre.in_channels},F], got {tuple(x.shape)}")
        if lengths is not None:
            if _wants_grad(x, self):
                raise NotImplementedError("ragged batches are an inference feature: call under torch.no_grad()")
            ln = torch.as_tensor(lengths).to(device=x.device, dtype=torch.int32).contiguous()
            if ln.shape != (x.shape[0],) or int(ln.min()) < 1 or int(ln.max()) > x.shape[2]:
                raise ValueError("lengths must be [B] frame counts within [1, F]")
            # frames past an item's end must read as zero padding at conv_pre's input
            mask = torch.arange(x.shape[2], device=x.device)[None, None, :] < ln[:, None, None]
            return self._engine(x.device).forward(x * mask, lengths=ln).clone()
        if _wants_grad(x, self):
            # differentiable call (an UPSTREAM-style `loss.backward()` loop): one autograd.Function over the training
            # forward (every conv input kept) and the hand-written backward — autograd.py
            from . import autograd
            return autograd.generator_forward(self, x)
        return self._engine(x.device).forward(x).clone()

    def _drop_engines(self):
        self.__dict__["_hg_engines"] = {}
        self.__dict__.pop("_hg_autograd", None)

    def remove_weight_norm(self):
        print('Removing weight norm...')
        for m in self.ups:
            remove_weight_norm(m)
        for blk in self.resblocks:
            blk.remove_weight_norm()
        remove_weight_norm(self.conv_pre)
        remove_weight_norm(self.conv_post)
        self._drop_engines()

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._drop_engines()
        return out


# --------------------------------------------------------------------------------------------------
# Discriminators (reference src/models.py:128-248).  Same module tree / state_dict keys as the reference; the
# forward pass runs on libhifigan_b200.so: Cin = 1 and Cout = 1 ends on CUDA-core kernels (hg_disc_*), every
# wide layer on the tcgen05 implicit-GEMM kernel (hg_conv1d_general_fwd) — strided layers through residue
# boxes, grouped layers as per-group N tiles (narrow groups merged into block-diagonal 32-wide ones).
# Activations live as bf16 [B*period][rows][C]: one independent 1-D sequence per period column.  Every call, with or
# without autograd recording, runs on the module's engine (autograd.py: _SubDiscTrainer.forward_single), so a
# discriminator computes the same numbers in both modes.
# --------------------------------------------------------------------------------------------------
def _round_up(n: int, m: int) -> int:
    return (n + m - 1) // m * m


class _DiscLayer:
    """One wide discriminator conv in GEMM-ready form (taps in the kernel's residue order, narrow groups
    merged into block-diagonal tiles)."""

    def __init__(self, cin, cout, k, stride, pad, groups):
        self.cin, self.cout, self.k, self.stride, self.pad = cin, cout, k, stride, pad
        cin_g, cout_g = cin // groups, cout // groups
        merge = 1
        if groups == 1:
            if cin % 32 or cout % 32:
                raise NotImplementedError(f"conv {cin}->{cout}: channel counts must be multiples of 32")
        else:
            while (cin_g * merge) % 32 or (cout_g * merge) not in (32, 64, 128, 256):
                merge *= 2
                if merge > groups:
                    raise NotImplementedError(f"cannot tile conv {cin}->{cout} groups={groups}")
        self.groups, self.merge = groups, merge
        self.groups_eff = groups // merge
        self.cin_tile = cin if groups == 1 else cin_g * merge
        order = (c_int * k)()
        _lib.check(_lib.lib().hg_conv1d_tap_order(k, stride, pad, order), "hg_conv1d_tap_order")
        self.order = list(order)

    def pack(self, w: torch.Tensor) -> torch.Tensor:
        """w fp32 contiguous [cout][cin/groups][k] on the device -> bf16 [k (kernel order)][cout][cin_tile]
        (hg_pack_disc_weight)."""
        out = torch.empty(self.k, self.cout, self.cin_tile, dtype=torch.bfloat16, device=w.device)
        _lib.check(_lib.lib().hg_pack_disc_weight(w.data_ptr(), self.cout, self.cin, self.groups, self.merge, self.k,
                                                  self.stride, self.pad, out.data_ptr(), 0, _stream()),
                   "hg_pack_disc_weight")
        return out


class _SubDiscriminator(torch.nn.Module):
    """forward() of DiscriminatorP / DiscriminatorS: y fp32 [B,1,T] -> (logits [B, H*p], feature maps fp32
    [B,C,H,p])."""

    def forward(self, x):
        _require_cuda(x, f"{type(self).__name__}.forward")
        from . import autograd
        return autograd.disc_forward(self, x, _wants_grad(x, self))


class DiscriminatorP(_SubDiscriminator):
    def __init__(self, period, kernel_size=5, stride=3, use_spectral_norm=False):
        super().__init__()
        self.period = period
        norm_f = spectral_norm if use_spectral_norm else _wn
        widths = [1, 32, 128, 512, 1024]
        layers = [norm_f(Conv2d(ci, co, (kernel_size, 1), (stride, 1), padding=(get_padding(5, 1), 0)))
                  for ci, co in zip(widths[:-1], widths[1:])]
        layers.append(norm_f(Conv2d(1024, 1024, (kernel_size, 1), 1, padding=(2, 0))))
        self.convs = nn.ModuleList(layers)
        self.conv_post = norm_f(Conv2d(1024, 1, (3, 1), 1, padding=(1, 0)))


class MultiPeriodDiscriminator(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.discriminators = nn.ModuleList([DiscriminatorP(p) for p in (2, 3, 5, 7, 11)])

    def forward(self, y, y_hat):
        y_d_rs, y_d_gs, fmap_rs, fmap_gs = [], [], [], []
        for d in self.discriminators:
            y_d_r, fmap_r = d(y)
            y_d_g, fmap_g = d(y_hat)
            y_d_rs.append(y_d_r); fmap_rs.append(fmap_r)
            y_d_gs.append(y_d_g); fmap_gs.append(fmap_g)
        return y_d_rs, y_d_gs, fmap_rs, fmap_gs


class DiscriminatorS(_SubDiscriminator):
    _SPEC = [(1, 128, 15, 1, 1, 7), (128, 128, 41, 2, 4, 20), (128, 256, 41, 2, 16, 20),
             (256, 512, 41, 4, 16, 20), (512, 1024, 41, 4, 16, 20), (1024, 1024, 41, 1, 16, 20),
             (1024, 1024, 5, 1, 1, 2)]

    def __init__(self, use_spectral_norm=False):
        super().__init__()
        norm_f = spectral_norm if use_spectral_norm else _wn
        self.convs = nn.ModuleList([norm_f(Conv1d(ci, co, k, s, groups=g, padding=p))
                                    for ci, co, k, s, g, p in self._SPEC])
        self.conv_post = norm_f(Conv1d(1024, 1, 3, 1, padding=1))

    def forward(self, x):
        out, fmap = super().forward(x)
        return out, [f.squeeze(-1) for f in fmap]   # [B,C,T,1] -> the reference's [B,C,T]


def _avgpool(x: torch.Tensor) -> torch.Tensor:
    """AvgPool1d(4, 2, padding=2) over the last dimension (hg_avgpool_4_2_2_fwd): [..., T] -> fp32 [..., T // 2 + 1]"""
    t = x.shape[-1]
    xin = x.detach().reshape(-1, t).contiguous().float()
    out = torch.empty(*x.shape[:-1], t // 2 + 1, dtype=torch.float32, device=x.device)
    _lib.check(_lib.lib().hg_avgpool_4_2_2_fwd(xin.data_ptr(), xin.shape[0], t, out.data_ptr(), _stream()),
               "hg_avgpool_4_2_2_fwd")
    return out


class MultiScaleDiscriminator(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.discriminators = nn.ModuleList([DiscriminatorS(use_spectral_norm=True), DiscriminatorS(),
                                             DiscriminatorS()])
        # kept for state_dict / attribute parity; the pooling itself runs in hg_avgpool_4_2_2_fwd
        self.meanpools = nn.ModuleList([AvgPool1d(4, 2, padding=2), AvgPool1d(4, 2, padding=2)])

    @staticmethod
    def _pool(x: torch.Tensor) -> torch.Tensor:
        if torch.is_grad_enabled() and x.requires_grad:
            from . import autograd
            return autograd.avgpool(x)
        return _avgpool(x)

    def forward(self, y, y_hat):
        _require_cuda(y, "MultiScaleDiscriminator.forward")
        _require_cuda(y_hat, "MultiScaleDiscriminator.forward")
        y_d_rs, y_d_gs, fmap_rs, fmap_gs = [], [], [], []
        for i, d in enumerate(self.discriminators):
            if i != 0:
                y, y_hat = self._pool(y), self._pool(y_hat)
            y_d_r, fmap_r = d(y)
            y_d_g, fmap_g = d(y_hat)
            y_d_rs.append(y_d_r); fmap_rs.append(fmap_r)
            y_d_gs.append(y_d_g); fmap_gs.append(fmap_g)
        return y_d_rs, y_d_gs, fmap_rs, fmap_gs


def _loss_mean(a32: torch.Tensor, b32: Optional[torch.Tensor], mode: int, c: float) -> torch.Tensor:
    """mean |a - b| (mode 0) or mean (c - a)^2 (mode 1) of contiguous fp32 device tensors (hg_loss_sum)"""
    acc = torch.zeros(1, dtype=torch.float32, device=a32.device)
    _lib.check(_lib.lib().hg_loss_sum(a32.data_ptr(), 0 if b32 is None else b32.data_ptr(), a32.numel(), mode, c,
                                      acc.data_ptr(), _stream()), "hg_loss_sum")
    return acc[0] / a32.numel()


def _device_mean(a: torch.Tensor, b: Optional[torch.Tensor], mode: int, c: float) -> torch.Tensor:
    """mean |a-b| (mode 0) or mean (c-a)^2 (mode 1) through hg_loss_sum; differentiable (hg_loss_grad) when an
    argument carries autograd history.  No CPU path."""
    if not a.is_cuda or (b is not None and not b.is_cuda):
        raise RuntimeError("hifigan_b200 losses have no CPU path; move the tensors to a B200")
    if torch.is_grad_enabled() and (a.requires_grad or (b is not None and b.requires_grad)):
        from . import autograd
        return autograd.device_mean(a, b, mode, c)
    return _loss_mean(a.detach().contiguous().float(), None if b is None else b.detach().contiguous().float(), mode, c)


def feature_loss(fmap_r, fmap_g):
    """2 * sum of mean |r - g| over all feature maps; reference src/models.py:251-257."""
    total = 0
    for maps_r, maps_g in zip(fmap_r, fmap_g):
        for r, g in zip(maps_r, maps_g):
            total = total + _device_mean(r, g, 0, 0.0)
    return total * 2


def discriminator_loss(disc_real_outputs, disc_generated_outputs):
    """LSGAN discriminator loss; per-sub-discriminator floats for logging; reference :260-271.
    The 2*N scalars cross to the host in ONE transfer instead of the reference's 2*N `.item()` syncs."""
    total, parts = 0, []
    for dr, dg in zip(disc_real_outputs, disc_generated_outputs):
        r_loss = _device_mean(dr, None, 1, 1.0)
        g_loss = _device_mean(dg, None, 1, 0.0)
        total = total + (r_loss + g_loss)
        parts += [r_loss.detach(), g_loss.detach()]
    host = torch.stack(parts).tolist() if parts else []
    return total, host[0::2], host[1::2]


def generator_loss(disc_outputs):
    """LSGAN generator loss; returns (sum, [per-sub-discriminator tensors]); reference :274-282."""
    gen_losses = [_device_mean(dg, None, 1, 1.0) for dg in disc_outputs]
    total = 0
    for l in gen_losses:
        total = total + l
    return total, gen_losses
