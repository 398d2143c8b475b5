"""SDE-DPM-Solver++(2M) (Lu et al., 2022, "DPM-Solver++: Fast Solver for Guided Sampling of Diffusion Probabilistic
Models", the second-order multistep solver of the reverse diffusion SDE with data prediction; the `sde-dpmsolver++`
of diffusers), restated in its textbook form on top of oracle/uvit_oracle.py: the schedule comes from its
ddpm_schedule, the grid from its ddim_timesteps, and the model is any callable (x, t, y) -> out, such as
uvit_oracle.uvit_forward or guidance_oracle.guided_model.  Nothing here reads the product's coefficient table.

With alpha_t = sqrt(abar_t), sigma_t = sqrt(1 - abar_t), lambda_t = log(alpha_t / sigma_t) and the data prediction
x0(x, t) = (x - sigma_t * eps) / alpha_t (predict_noise) or the model output itself (predict_original), the step
from t to the next grid point s with h = lambda_s - lambda_t is
    order 1:  D = x0_t
    order 2:  r = h_prev / h,  D = (1 + 1/(2r)) x0_t - 1/(2r) x0_prev
    x_s = (sigma_s / sigma_t) exp(-h) x + alpha_s (1 - exp(-2h)) D + sigma_s sqrt(1 - exp(-2h)) z
with z the noise of the step at t, and no noise on the final step (s = 0), as in the DDIM branch.  The first and the
final step are order 1, the others order 2.  The hand-off between backbones is the DDIM branch's: after the step at
t, `if t < 1000 - t_switch: model = late`.

Coefficients are fp64 Python floats from the fp32 schedule.  x keeps its dtype: an fp64 x_T gives an fp64 run."""
from __future__ import annotations

import math

import torch

from oracle import uvit_oracle as O


def _lambda(abar: float) -> float:
    return math.log(math.sqrt(abar)) - math.log(math.sqrt(1 - abar))


def steps(n: int, all_first_order: bool = False) -> list:
    """Per step of the n-point grid: dict(t, s, alpha_t, sigma_t, alpha_s, sigma_s, h, r, order) in fp64 (r is None
    for the first step)."""
    ab = [float(v) for v in O.ddpm_schedule()["alphas_bar"]]
    ts = O.ddim_timesteps(n)
    evals = len(ts) - 1
    out, h_prev = [], None
    for k, (t, s) in enumerate(zip(ts[:-1], ts[1:])):
        h = _lambda(ab[s]) - _lambda(ab[t])
        order = 1 if all_first_order or k == 0 or k == evals - 1 else 2
        out.append(dict(t=t, s=s, alpha_t=math.sqrt(ab[t]), sigma_t=math.sqrt(1 - ab[t]), alpha_s=math.sqrt(ab[s]),
                        sigma_s=math.sqrt(1 - ab[s]), h=h, r=None if h_prev is None else h_prev / h, order=order))
        h_prev = h
    return out


def step(st: dict, x, out, x0_prev, z, rule: str = "predict_noise"):
    """One step of the solver from st["t"] to st["s"]; returns (x_s, x0_t)."""
    x0 = (x - st["sigma_t"] * out) / st["alpha_t"] if rule == "predict_noise" else out
    if st["order"] == 1:
        d = x0
    else:
        r = st["r"]
        d = (1 + 1 / (2 * r)) * x0 - (1 / (2 * r)) * x0_prev
    h = st["h"]
    x = (st["sigma_s"] / st["sigma_t"]) * math.exp(-h) * x + st["alpha_s"] * (1 - math.exp(-2 * h)) * d
    if st["s"] > 0:
        x = x + st["sigma_s"] * math.sqrt(1 - math.exp(-2 * h)) * z
    return x, x0


def sample_sde_dpm_solver(early, late, t_switch, x_T: torch.Tensor, n: int, noise, y=None,
                          rule: str = "predict_noise", trace: dict | None = None,
                          all_first_order: bool = False) -> torch.Tensor:
    """SDE-DPM-Solver++(2M) over the n-point DDIM grid (n - 1 model evaluations); returns x at t = 0.  noise: a
    tensor indexed by t or a callable t -> z.  all_first_order makes every step first order (the DDPM posterior step
    between grid points)."""
    if rule not in ("predict_noise", "predict_original"):
        raise ValueError(f"SDE-DPM-Solver++ needs a noise or data prediction, not {rule!r}")
    x, model, x0_prev = x_T, early, None
    for st in steps(n, all_first_order):
        t = st["t"]
        with torch.no_grad():
            out = model(x, t * torch.ones(x.shape[0], device=x.device), y)
        z = None
        if st["s"] > 0:
            z = noise(t) if callable(noise) else noise[t]
        if trace is not None:
            trace.setdefault("t", []).append(t)
            trace.setdefault("late", []).append(model is late)
            trace.setdefault("out", []).append(out)
        x, x0_prev = step(st, x, out, x0_prev, z, rule)
        if late is not None and t < 1000 - t_switch:
            model = late
    return x
