"""The reference of the training step's gradient guard (h.clip_grad_norm), for the tests: the fork's
manual-optimisation callback (manual_optimization_callback.py:23-36) written over torch,

    total = torch.nn.utils.clip_grad_norm_(params_N, max_norm)
    if torch.isfinite(total): optim_N.step()

as an optimizer wrapper that oracle/train_oracle.train_step drives like a plain torch.optim.AdamW (it calls only
zero_grad() and step()).  params_N are ALL of the wrapped optimizer's parameters: for D that is
chain(msd.parameters(), mpd.parameters()), as for UPSTREAM's optim_d."""
import torch

from oracle import train_oracle as TO


class ClipSkip:
    """torch.optim optimizer + the callback's rule; `norms` holds the totals clip_grad_norm_ returned, one per step"""

    def __init__(self, opt, max_norm: float):
        self.opt, self.max_norm = opt, max_norm
        self.param_groups = opt.param_groups
        self.state = opt.state
        self.norms = []
        self.skipped = 0

    def zero_grad(self):
        self.opt.zero_grad()

    def step(self):
        params = [p for group in self.opt.param_groups for p in group["params"]]
        total = torch.nn.utils.clip_grad_norm_(params, self.max_norm)
        self.norms.append(float(total))
        if torch.isfinite(total):
            self.opt.step()
        else:
            self.skipped += 1


def make_guarded_optimizers(sd_g, sd_mpd, sd_msd, h, max_norm: float):
    """UPSTREAM's (optim_g, optim_d) of oracle/train_oracle.make_optimizers, each wrapped in ClipSkip"""
    og, od = TO.make_optimizers(sd_g, sd_mpd, sd_msd, h)
    return ClipSkip(og, max_norm), ClipSkip(od, max_norm)


def guarded_train_step(sd_g, sd_mpd, sd_msd, h, x, y, y_mel, optims):
    """oracle/train_oracle.train_step under the guard; `losses` gains "grad_norm_g" / "grad_norm_d" (the totals torch
    returned for this step).  optims = make_guarded_optimizers(...), kept across steps."""
    out = TO.train_step(sd_g, sd_mpd, sd_msd, h, x, y, y_mel, optims=optims)
    out[0]["grad_norm_g"], out[0]["grad_norm_d"] = optims[0].norms[-1], optims[1].norms[-1]
    return out
