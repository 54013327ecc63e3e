"""The reference of the gradient guard (tests/grad_guard_ref.py: the training oracle's step under
torch.nn.utils.clip_grad_norm_ and the skip of a non-finite step), which the GPU tests of the in-graph guard compare
against, pinned on the CPU against a hand-written torch loop of the fork's manual-optimisation callback: clip every gradient of the optimizer by min(1, max_norm / (total + 1e-6)), then step
only if the pre-clip norm is finite.  A small generator (the tiny topology, upsampling 256x) keeps it fast."""
import copy

import torch

from oracle import hifigan_oracle as O
from oracle import train_oracle as TO
from grad_guard_ref import guarded_train_step, make_guarded_optimizers


class HandGuard:
    """optimizer wrapper: the callback's rule written out by hand (fp64 norm, explicit coefficient)"""

    def __init__(self, opt, max_norm):
        self.opt, self.max_norm, self.norms, self.skipped = opt, max_norm, [], 0
        self.param_groups = opt.param_groups

    def zero_grad(self):
        self.opt.zero_grad()

    def step(self):
        ps = [p for g in self.opt.param_groups for p in g["params"]]
        total = float(torch.sqrt(sum((p.grad.double() ** 2).sum() for p in ps)))
        self.norms.append(total)
        if not torch.isfinite(torch.tensor(total)):
            self.skipped += 1
            return
        coef = min(1.0, self.max_norm / (total + 1e-6))
        for p in ps:
            p.grad.mul_(coef)
        self.opt.step()


def _setup():
    h = O.config("tiny")
    h.update(upsample_rates=[8, 8, 4], upsample_kernel_sizes=[16, 16, 8])        # 256x: the mel hop
    import hifigan_b200 as H
    torch.manual_seed(3)
    nets = (H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator())
    sds = [{k: v.detach().clone() for k, v in m.state_dict().items()} for m in nets]
    ya = O.synthetic_audio(2, 2048, seed=8)
    mel = lambda a, fmax: O.mel_spectrogram(a, 1024, 80, 22050, 256, 1024, 0, fmax)
    return h, sds, ya, mel


def _run(h, sds, batches, guard):
    """guard: ("ref", max_norm) (grad_guard_ref) or ("hand", max_norm); returns (state dicts, optimizers, losses)"""
    sd = [TO.leaf_params(copy.deepcopy(s)) for s in sds]
    kind, max_norm = guard
    if kind == "ref":
        optims = make_guarded_optimizers(*sd, h, max_norm)
        losses = [guarded_train_step(*sd, h, x, y, y_mel, optims)[0] for x, y, y_mel in batches]
    else:
        og, od = TO.make_optimizers(*sd, h)
        optims = (HandGuard(og, max_norm), HandGuard(od, max_norm))
        losses = [TO.train_step(*sd, h, x, y, y_mel, optims=optims)[0] for x, y, y_mel in batches]
    return sd, optims, losses


def _moments(opt, sd, keys):
    return {k: opt.state[sd[k]] for k in keys if sd[k] in opt.state}


def test_oracle_guard_clips_and_skips_like_the_callback():
    torch.set_num_threads(max(1, torch.get_num_threads()))
    h, sds, ya, mel = _setup()
    x, y_mel = mel(ya, 8000), mel(ya, None)
    clean = (x, ya.unsqueeze(1), y_mel)
    bad_y = ya.clone()
    bad_y[1, 700] = float("nan")                     # one NaN in the real audio: the D gradient is NaN
    batches = [clean, clean, (x, bad_y.unsqueeze(1), y_mel), clean]
    # unclipped norms of step 1 set the limit: half of the smaller one, so both networks clip
    sd1 = [TO.leaf_params(copy.deepcopy(s)) for s in sds]
    ref1 = guarded_train_step(*sd1, h, *clean, make_guarded_optimizers(*sd1, h, float("inf")))[0]
    max_norm = 0.5 * min(ref1["grad_norm_g"], ref1["grad_norm_d"])
    sd_o, (og, od), lo = _run(h, sds, batches, ("ref", max_norm))
    sd_h, (hg, hd), lh = _run(h, sds, batches, ("hand", max_norm))
    # the reference reports the totals torch returned; they match the hand-computed fp64 norms and exceed the limit
    for i in range(len(batches)):
        for name, hand in (("grad_norm_g", hg), ("grad_norm_d", hd)):
            got, ref = float(lo[i][name]), hand.norms[i]
            if i == 2 and name == "grad_norm_d":
                assert not torch.isfinite(torch.tensor(got)) and not torch.isfinite(torch.tensor(ref))
                continue
            if not torch.isfinite(torch.tensor(ref)):
                assert not torch.isfinite(torch.tensor(got)), (i, name, got)
                continue
            # torch's fp32 norm of a 5M-element tensor is itself off by ~4e-4 on the CPU (measured 1.01261 vs fp64 1.01302)
            assert abs(got - ref) <= 2e-3 * ref, (i, name, got, ref)
            if i == 0:
                assert got > 1.5 * max_norm, (name, got, max_norm)    # clipped: the limit is binding
    assert hd.skipped == 1
    # same trajectory: parameters and both moments of both networks, and torch's step counts (applied updates only)
    # (the coefficients differ by torch's fp32 norm error: each tensor's update and moments are compared as a whole)
    for sd_a, sd_b, sd0, opt_a, opt_b in ((sd_o[0], sd_h[0], sds[0], og.opt, hg.opt),
                                          (sd_o[1], sd_h[1], sds[1], od.opt, hd.opt),
                                          (sd_o[2], sd_h[2], sds[2], od.opt, hd.opt)):
        keys = [k for k, v in sd_a.items() if v.requires_grad]
        for k in keys:
            da, db = sd_a[k].detach() - sd0[k], sd_b[k].detach() - sd0[k]
            assert (da - db).norm() <= 2e-3 * db.norm(), k
        ma, mb = _moments(opt_a, sd_a, keys), _moments(opt_b, sd_b, keys)
        assert ma.keys() == mb.keys() and len(ma) == len(keys)
        for k in keys:
            for s in ("exp_avg", "exp_avg_sq"):
                assert (ma[k][s] - mb[k][s]).norm() <= 2e-3 * mb[k][s].norm(), (k, s)
            assert float(ma[k]["step"]) == float(mb[k]["step"])
    d_steps = {float(od.state[p]["step"]) for g in od.param_groups for p in g["params"]}
    assert d_steps == {3.0} and od.skipped == 1      # 4 steps, the NaN one skipped


def test_oracle_guard_skip_leaves_the_optimizer_state_untouched():
    """a skipped D step keeps parameters, moments and the step count bit for bit"""
    h, sds, ya, mel = _setup()
    x, y_mel = mel(ya, 8000), mel(ya, None)
    sd = [TO.leaf_params(copy.deepcopy(s)) for s in sds]
    optims = make_guarded_optimizers(*sd, h, 1.0)
    guarded_train_step(*sd, h, x, ya.unsqueeze(1), y_mel, optims)
    od = optims[1]
    params = [p for g in od.param_groups for p in g["params"]]
    before = [(p.detach().clone(), od.state[p]["exp_avg"].clone(), od.state[p]["exp_avg_sq"].clone(),
               float(od.state[p]["step"])) for p in params]
    bad = ya.clone()
    bad[0, 10] = float("inf")
    losses = guarded_train_step(*sd, h, x, bad.unsqueeze(1), y_mel, optims)[0]
    assert not torch.isfinite(torch.tensor(losses["grad_norm_d"]))
    for p, (p0, m0, v0, s0) in zip(params, before):
        assert torch.equal(p.detach(), p0) and torch.equal(od.state[p]["exp_avg"], m0)
        assert torch.equal(od.state[p]["exp_avg_sq"], v0) and float(od.state[p]["step"]) == s0
