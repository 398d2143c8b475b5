"""Classifier-free guidance (fp32), restated on top of oracle/uvit_oracle.py: its forward, its DDPM / DDIM loops and
their update rules are reused unchanged; only the model callable differs.

The reference has no guidance, so no reference-made fixture can pin this module.  What it builds on is pinned:
the class-conditional forward by tests/golden/uvit_forward_tiny_cls.npz and the two sampling loops by
duodiff_sampler_tiny.npz / ddim_sampler_tiny.npz.  The guided step is U-ViT's form,
    eps = eps_c + s * (eps_c - eps_u),
eps_c with the caller's labels y and eps_u with the null label, both from ONE forward on the 2B rows [x ; x]; the
combination is three separately rounded fp32 operations (s = 0 gives eps_c)."""
from __future__ import annotations

import torch

from oracle import uvit_oracle as O


def combine(eps_c: torch.Tensor, eps_u: torch.Tensor, scale: float) -> torch.Tensor:
    """eps_c + s * (eps_c - eps_u): subtract, multiply, add, each rounded (what the CUDA tail computes)."""
    return eps_c + scale * (eps_c - eps_u)


def guided_model(model, scale: float, null_label: int):
    """(x, t, y) -> guided eps of `model` ((x, t, y) -> eps), from one forward on [x ; x], [t ; t], [y ; null]."""
    def f(x, t, y):
        B = x.shape[0]
        out = model(torch.cat([x, x]), torch.cat([t, t]), torch.cat([y, torch.full_like(y, int(null_label))]))
        return combine(out[:B], out[B:], scale)
    return f


def sample_ddpm_guided(early, late, t_switch, x_T: torch.Tensor, noise, y: torch.Tensor, scale: float,
                       null_label: int, rule: str = "predict_noise", t_first: int = 999, t_last: int = 0,
                       trace: dict | None = None) -> torch.Tensor:
    """O.sample_ddpm with both backbones guided; `trace` records the guided eps per step."""
    return O.sample_ddpm(guided_model(early, scale, null_label),
                         guided_model(late, scale, null_label) if late is not None else None, t_switch, x_T, noise,
                         y=y, rule=rule, t_first=t_first, t_last=t_last, trace=trace)


def sample_ddim_guided(early, late, t_switch, x_T: torch.Tensor, noise, ddim_steps: int, eta: float, y: torch.Tensor,
                       scale: float, null_label: int, trace: dict | None = None,
                       n_pairs: int | None = None) -> torch.Tensor:
    """O.sample_ddim with both backbones guided."""
    return O.sample_ddim(guided_model(early, scale, null_label),
                         guided_model(late, scale, null_label) if late is not None else None, t_switch, x_T, noise,
                         ddim_steps, eta, y=y, trace=trace, n_pairs=n_pairs)
