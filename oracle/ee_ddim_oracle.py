"""ORACLE — test infrastructure only.  Never imported by the product path (duodiff_b200/).

DDIM sampling with early exit: the DeeDiff / AdaDiff selection of eesampler.py:57-72 (uvit_oracle.ee_forward +
ee_select) at every step of the strided DDIM loop of sampler.py:103-126 (uvit_oracle.ddim_step, including the
reference's sigma_t^2 * z noise term).  The reference has no such loop; this composes two of its pinned pieces.
"""
from __future__ import annotations

import torch

from oracle.uvit_oracle import ddim_step, ddim_timesteps, ddpm_schedule, ee_select


def ee_sample_ddim(ee_model, threshold: float, depth: int, x_T: torch.Tensor, noise, ddim_steps: int, eta: float,
                   y=None, trace: dict | None = None):
    """-> (x_0, error_prediction_by_timestep [1000, depth], indices_by_timestep [1000, B]).

    ``ee_model`` is a callable (x, timesteps, y) -> (eps_full, [cls_i], [out_i]) like uvit_oracle.ee_forward.  The
    logs are indexed by t; rows of timesteps the grid does not visit are NaN.  ``noise`` as in uvit_oracle.sample_ddim
    (a tensor indexed by t or a callable t -> z; z = 0 for the last step, s == 0).  ``trace`` (tests): per step the input
    x_t and the per-sample probe outputs [depth+1, B], keyed by t, as in uvit_oracle.ee_sample."""
    sch = ddpm_schedule(x_T.device)
    B = x_T.shape[0]
    err_log = torch.full((1000, depth), float("nan"))
    idx_log = torch.full((1000, B), float("nan"))
    ts = ddim_timesteps(ddim_steps)
    x = x_T
    for t, s in zip(ts[:-1], ts[1:]):
        time_tensor = t * torch.ones(B, device=x.device)
        with torch.no_grad():
            eps_full, cls, outs = ee_model(x, time_tensor, y)
        eps, indices, scores = ee_select(eps_full, cls, outs, threshold)
        err_log[t] = scores.mean(axis=1)[:depth].cpu()
        idx_log[t, :] = indices.cpu().float()
        if trace is not None:
            trace.setdefault("x_in", {})[t] = x
            trace.setdefault("scores", {})[t] = scores
        z = None
        if s > 0:
            z = noise(t) if callable(noise) else noise[t]
        x = ddim_step(sch, eps, x, t, s, eta, z)
    return x, err_log, idx_log
