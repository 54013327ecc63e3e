"""The single-layer weight-preparation entry points against the batched job bodies they share.

Each C entry point (hg_pack_conv1d_weight, hg_pack_convtr1d_weight, hg_pack_dgrad_weight, hg_pack_disc_weight,
hg_wgrad_finish_conv, hg_unpack_wgrad_conv, hg_weight_norm_bwd) is run next to the same job built the way the
trainers build it (batched.JobTable, hg_prep_batched), on seeded inputs at the models' shapes.  The two must agree
bit for bit: the standalone / per-layer paths and the batched training paths compute the same numbers."""
import json
import os
from ctypes import byref, c_int

import pytest
import torch

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


def _rand(gen, *shape):
    return torch.randn(*shape, generator=gen).cuda()


def _run_job(kind, nblocks, smem=0, **kw):
    from hifigan_b200 import batched
    t = batched.JobTable(torch.device("cuda"))
    t.add("p", kind, nblocks, smem, **kw)
    t.finalize().launch("p")
    torch.cuda.synchronize()


def _config(ver):
    with open(os.path.join(ROOT, "hifi-gan_b200", "configs", f"config_{ver}.json")) as f:
        return json.load(f)


def _gen_shapes(ver):
    """(cin, cout, k) of conv_pre and every ResBlock conv; (cin, cout, k, stride, padding) of every upsampling layer"""
    h = _config(ver)
    c0 = h["upsample_initial_channel"]
    convs, ups = {(h.get("num_mels", 80), c0, 7)}, []
    for i, (u, k) in enumerate(zip(h["upsample_rates"], h["upsample_kernel_sizes"])):
        cin, cout = c0 // 2 ** i, c0 // 2 ** (i + 1)
        ups.append((cin, cout, k, u, (k - u) // 2))
        convs |= {(cout, cout, rk) for rk in h["resblock_kernel_sizes"]}
    return sorted(convs), ups


# wide discriminator layers: cin, cout, k, stride, pad, groups (MPD: (5, 1) kernels run as 1-D; MSD: grouped, k = 41)
DISC_LAYERS = [
    (32, 128, 5, 3, 2, 1), (128, 512, 5, 3, 2, 1), (512, 1024, 5, 3, 2, 1), (1024, 1024, 5, 1, 2, 1),
    (128, 128, 41, 2, 20, 4), (128, 256, 41, 2, 20, 16), (256, 512, 41, 4, 20, 16), (512, 1024, 41, 4, 20, 16),
    (1024, 1024, 41, 1, 20, 16), (1024, 1024, 5, 1, 2, 1),
]


@pytest.mark.parametrize("ver", ["v1", "v2", "v3"])
@pytest.mark.parametrize("weight_norm", [True, False])
def test_generator_conv_pack(H, ver, weight_norm):
    """hg_pack_conv1d_weight on the zero-padded parameters (_PackedConv.refresh) == HG_JOB_GEN_CONV on the raw ones
    (_PackedConv.add_pack_job), including V2's padded 8-channel stage"""
    from hifigan_b200 import _lib, batched
    from hifigan_b200.models import _pad_ch
    L = _lib.lib()
    for cin, cout, k in _gen_shapes(ver)[0]:
        gen = torch.Generator().manual_seed(cin * 1000 + cout * 10 + k)
        cin_p, cout_p = _pad_ch(cin), _pad_ch(cout)
        v = _rand(gen, cout, cin, k)
        g = (torch.rand(cout, generator=gen) + 0.5).cuda() if weight_norm else None
        vp = torch.cat([v, v.new_zeros(cout_p - cout, cin, k)]).contiguous()
        gp = None if g is None else torch.cat([g, g.new_zeros(cout_p - cout)])
        w_one = torch.full((k, cout_p, cin_p), 7.0, dtype=torch.bfloat16, device="cuda")
        w_job = w_one.clone()
        _lib.check(L.hg_pack_conv1d_weight(vp.data_ptr(), 0 if gp is None else gp.data_ptr(), cout_p, cin, k, cin_p,
                                           w_one.data_ptr(), _st()), "hg_pack_conv1d_weight")
        _run_job(batched.GEN_CONV, cout_p, src0=v, src1=g, dst0=w_job, ints=(cout, cin, k, cout_p, cin_p))
        assert torch.equal(w_one, w_job), (ver, cin, cout, k)


@pytest.mark.parametrize("ver", ["v1", "v2", "v3"])
def test_generator_convtr_pack(H, ver):
    """hg_pack_convtr1d_weight (caller-padded) == HG_JOB_GEN_CONVTR for every upsampling layer of each config"""
    from hifigan_b200 import _lib, batched
    from hifigan_b200.models import _pad_ch
    L = _lib.lib()
    for cin, cout, k, u, pad in _gen_shapes(ver)[1]:
        gen = torch.Generator().manual_seed(cin + cout + k + u)
        nshift, smin = c_int(), c_int()
        _lib.check(L.hg_convtr1d_geometry(k, u, pad, byref(nshift), byref(smin)))
        cin_p, cout_p = _pad_ch(cin), _pad_ch(cout)
        v = _rand(gen, cin, cout, k)
        g = (torch.rand(cin, generator=gen) + 0.5).cuda()
        vp = v.new_zeros(cin_p, cout_p, k)
        vp[:cin, :cout] = v
        gp = torch.cat([g, g.new_zeros(cin_p - cin)])
        w_one = torch.full((nshift.value, u * cout_p, cin_p), 7.0, dtype=torch.bfloat16, device="cuda")
        w_job = w_one.clone()
        _lib.check(L.hg_pack_convtr1d_weight(vp.data_ptr(), gp.data_ptr(), cin_p, cout_p, k, u, pad, w_one.data_ptr(),
                                             _st()), "hg_pack_convtr1d_weight")
        _run_job(batched.GEN_CONVTR, cin_p, src0=v, src1=g, dst0=w_job,
                 ints=(cin, cout, k, cin_p, cout_p, u, pad, nshift.value, smin.value))
        assert torch.equal(w_one, w_job), (ver, cin, cout, k)


@pytest.mark.parametrize("ver", ["v1", "v2", "v3"])
def test_dgrad_bank_transpose(H, ver):
    """hg_pack_dgrad_weight == HG_JOB_TRANSPOSE_TILE (_GenLayerGrad.add_jobs) on Generator forward banks, polyphase
    upsampling banks included"""
    from hifigan_b200 import _lib, batched
    from hifigan_b200.models import _pad_ch
    L = _lib.lib()
    convs, ups = _gen_shapes(ver)
    banks = [(k, _pad_ch(cout), _pad_ch(cin)) for cin, cout, k in convs]
    for cin, cout, k, u, pad in ups:
        nshift, smin = c_int(), c_int()
        _lib.check(L.hg_convtr1d_geometry(k, u, pad, byref(nshift), byref(smin)))
        banks.append((nshift.value, u * _pad_ch(cout), _pad_ch(cin)))
    for taps, rows, c in banks:
        gen = torch.Generator().manual_seed(taps * 7 + rows + c)
        w = _rand(gen, taps, rows, c).bfloat16()
        out_one = torch.full((taps, c, rows), 7.0, dtype=torch.bfloat16, device="cuda")
        out_job = out_one.clone()
        _lib.check(L.hg_pack_dgrad_weight(w.data_ptr(), taps, rows, c, out_one.data_ptr(), _st()),
                   "hg_pack_dgrad_weight")
        tc, tn = (c + 31) // 32, (rows + 31) // 32
        _run_job(batched.TRANSPOSE_TILE, taps * tc * tn, 32 * 34 * 2, src0=w, dst0=out_job,
                 ints=(taps, rows, c, tc, tn))
        assert torch.equal(out_one, out_job), (ver, taps, rows, c)


@pytest.mark.parametrize("case", DISC_LAYERS)
def test_disc_forward_and_dgrad_banks(H, case):
    """hg_pack_disc_weight (w_fwd, and w_dgrad where the shape tiles) == the _DiscSlot jobs: HG_JOB_DISC_ROW with the
    weight_norm fold (its effective weight feeds the entry point) and with g NULL (the spectral-norm slots), and
    HG_JOB_DISC_DGRAD_TILE"""
    from hifigan_b200 import _lib, batched
    from hifigan_b200.models import _DiscLayer
    L = _lib.lib()
    cin, cout, k, s, pad, groups = case
    layer = _DiscLayer(cin, cout, k, s, pad, groups)
    cin_g, cout_g = cin // groups, cout // groups
    gen = torch.Generator().manual_seed(sum(case))
    v = _rand(gen, cout, cin_g, k)
    g = (torch.rand(cout, generator=gen) + 0.5).cuda()
    ints = (cout, cin_g, k, layer.merge, cout_g, layer.cin_tile)
    eff = torch.empty(cout, cin_g, k, device="cuda")
    fwd_wn = torch.full((k, cout, layer.cin_tile), 7.0, dtype=torch.bfloat16, device="cuda")
    _run_job(batched.DISC_ROW, cout, cin_g * k * 4, src0=v, src1=g, dst0=eff, dst1=fwd_wn, ints=ints, tab=layer.order)
    fwd_sn = torch.full_like(fwd_wn, 7.0)
    _run_job(batched.DISC_ROW, cout, cin_g * k * 4, src0=eff, dst1=fwd_sn, ints=ints, tab=layer.order)
    fwd_one = torch.full_like(fwd_wn, 7.0)
    _lib.check(L.hg_pack_disc_weight(eff.data_ptr(), cout, cin, groups, layer.merge, k, s, pad, fwd_one.data_ptr(), 0,
                                     _st()), "hg_pack_disc_weight")
    torch.cuda.synchronize()
    assert torch.equal(fwd_one, fwd_wn) and torch.equal(fwd_one, fwd_sn)

    nshift, smin = c_int(), c_int()
    _lib.check(L.hg_convtr1d_geometry(k, s, pad, byref(nshift), byref(smin)))
    cout_tile = cout_g * layer.merge
    tci = 32 if k <= 10 else 8
    while tci > 2 and (cin_g % tci or cin % tci):
        tci >>= 1
    smem = 32 * (tci * k + 1) * 4
    assert cin_g % tci == 0 and cin % tci == 0 and cout_tile % 32 == 0 and smem <= 48 * 1024   # the tiled job
    dg_one = torch.full((nshift.value, s * cin, cout_tile), 7.0, dtype=torch.bfloat16, device="cuda")
    dg_job = dg_one.clone()
    _lib.check(L.hg_pack_disc_weight(eff.data_ptr(), cout, cin, groups, layer.merge, k, s, pad, 0, dg_one.data_ptr(),
                                     _st()), "hg_pack_disc_weight")
    _run_job(batched.DISC_DGRAD_TILE, (cin // tci) * (cout_tile // 32), smem, src0=eff, dst0=dg_job,
             ints=(cout, cin_g, k, layer.merge, cout_g, cin, s, pad, nshift.value, smin.value, cout_tile, tci,
                   cin // tci))
    assert torch.equal(dg_one, dg_job)


def _finish_conv_ints(layer, cin_g, accumulate):
    return (0, layer.cout, cin_g, layer.k, layer.cout, layer.cin_tile, layer.cout // layer.groups, layer.merge,
            0, 0, 0, 0, accumulate)


def _packed_pos(order):
    pos = [0] * len(order)
    for q, tap in enumerate(order):
        pos[tap] = q
    return pos


@pytest.mark.parametrize("case", DISC_LAYERS)
def test_wgrad_finish_and_unpack(H, case):
    """hg_wgrad_finish_conv (accumulate 0 / 1, g NULL) and hg_unpack_wgrad_conv == HG_JOB_FINISH_ROW mode 0 on the
    packed weight gradient of a wide discriminator layer (non-identity tap order, merged groups)"""
    from hifigan_b200 import _lib, batched
    from hifigan_b200.models import _DiscLayer
    L = _lib.lib()
    cin, cout, k, s, pad, groups = case
    layer = _DiscLayer(cin, cout, k, s, pad, groups)
    cin_g = cin // groups
    gen = torch.Generator().manual_seed(sum(case) + 1)
    dwp = _rand(gen, k, cout, layer.cin_tile)
    v = _rand(gen, cout, cin_g, k)
    g = (torch.rand(cout, generator=gen) + 0.5).cuda()
    dv0, dg0 = _rand(gen, cout, cin_g, k), _rand(gen, cout)
    order = (c_int * k)(*layer.order)
    pos = _packed_pos(layer.order)
    for accumulate in (0, 1):
        for gg in (g, None):
            dv_one, dg_one = dv0.clone(), dg0.clone()
            dv_job, dg_job = dv0.clone(), dg0.clone()
            _lib.check(L.hg_wgrad_finish_conv(dwp.data_ptr(), cout, cin_g, k, cout, layer.cin_tile,
                                              cout // groups, layer.merge, order, v.data_ptr(),
                                              0 if gg is None else gg.data_ptr(), accumulate, dv_one.data_ptr(),
                                              dg_one.data_ptr(), _st()), "hg_wgrad_finish_conv")
            _run_job(batched.FINISH_ROW, cout, cin_g * k * 4, src0=dwp, src1=gg, src2=v, dst0=dv_job, dst1=dg_job,
                     ints=_finish_conv_ints(layer, cin_g, accumulate), tab=pos)
            assert torch.equal(dv_one, dv_job) and torch.equal(dg_one, dg_job), (accumulate, gg is None)
    dw_one = torch.full((cout, cin_g, k), 7.0, device="cuda")
    dw_job = dw_one.clone()
    _lib.check(L.hg_unpack_wgrad_conv(dwp.data_ptr(), cout, cin_g, k, cout, layer.cin_tile, cout // groups,
                                      layer.merge, order, dw_one.data_ptr(), _st()), "hg_unpack_wgrad_conv")
    _run_job(batched.FINISH_ROW, cout, cin_g * k * 4, src0=dwp, dst0=dw_job,
             ints=_finish_conv_ints(layer, cin_g, 0), tab=pos)
    assert torch.equal(dw_one, dw_job)


@pytest.mark.parametrize("d0,d1,k", [(32, 1, 5), (128, 1, 15), (1, 1024, 3), (1, 32, 7), (40, 30, 7)])
def test_weight_norm_bwd(H, d0, d1, k):
    """hg_weight_norm_bwd on a dense gradient == HG_JOB_FINISH_ROW mode 0 on the same gradient in packed form (identity
    taps, one group): the discriminator ends' and conv_post's parameter gradients (_route_weight_grad)"""
    from hifigan_b200 import _lib, batched
    L = _lib.lib()
    gen = torch.Generator().manual_seed(d0 * 100 + d1 + k)
    dw = _rand(gen, d0, d1, k)
    v = _rand(gen, d0, d1, k)
    g = (torch.rand(d0, generator=gen) + 0.5).cuda()
    packed = dw.permute(2, 0, 1).contiguous()          # [k][d0][d1]
    dv0, dg0 = _rand(gen, d0, d1, k), _rand(gen, d0)
    for accumulate in (0, 1):
        dv_one, dg_one = dv0.clone(), dg0.clone()
        dv_job, dg_job = dv0.clone(), dg0.clone()
        _lib.check(L.hg_weight_norm_bwd(dw.data_ptr(), v.data_ptr(), g.data_ptr(), d0, d1 * k, accumulate,
                                        dv_one.data_ptr(), dg_one.data_ptr(), _st()), "hg_weight_norm_bwd")
        _run_job(batched.FINISH_ROW, d0, d1 * k * 4, src0=packed, src1=g, src2=v, dst0=dv_job, dst1=dg_job,
                 ints=(0, d0, d1, k, d0, d1, d0, 1, 0, 0, 0, 0, accumulate), tab=range(k))
        assert torch.equal(dv_one, dv_job) and torch.equal(dg_one, dg_job), accumulate
