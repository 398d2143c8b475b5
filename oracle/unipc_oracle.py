"""UniPC (Zhao et al., 2023, "UniPC: A Unified Predictor-Corrector Framework for Fast Sampling of Diffusion Models"),
variant bh2, order 2, data prediction, restated in its structured UniP / UniC form on top of oracle/uvit_oracle.py: the
schedule comes from its ddpm_schedule, the grid from its ddim_timesteps, and the model is any callable (x, t, y) -> out,
such as uvit_oracle.uvit_forward or guidance_oracle.guided_model.  Nothing here reads the product's coefficient table.

With alpha_t = sqrt(abar_t), sigma_t = sqrt(1 - abar_t), lambda_t = log(alpha_t / sigma_t) and the data prediction
D = (x - sigma_t * eps) / alpha_t (predict_noise) or the model output itself (predict_original), on the grid
t_0 > t_1 > ... > t_E (E = n - 1 model evaluations, the model runs at x_k, t_k):
    UniC (k >= 1, order p_{k-1}), from the previous base point xc_{k-1} to t_k, with the uncorrected x_k's D_k:
        h = lambda_k - lambda_{k-1},  B = expm1(-h)
        xc_k = (sigma_k / sigma_{k-1}) xc_{k-1} - alpha_k expm1(-h) D_{k-1}
               - alpha_k B (sum_i rho_i (D_{k-1-i} - D_{k-1}) / r_i + rho_last (D_k - D_{k-1}))
        with r_i = (lambda_{k-1-i} - lambda_{k-1}) / h and rho solving the order conditions below; order 1: rho = [1/2]
    UniP (order p_k), from xc_k to t_{k+1}:
        xhat = (sigma_{k+1} / sigma_k) xc_k - alpha_{k+1} expm1(-h') D_k - alpha_{k+1} B' (1/2) (D_{k-1} - D_k) / r'
        (the last term on order 2 only)
p_k = 1 for the first and the final step (lower_order_final), 2 otherwise; xc_0 = x_0 (no corrector at k = 0).
The order conditions (UniPC's bh update): R[i][j] = r_j^i, b[i] = h phi_{i+1}(h) (i + 1)! / B with h phi_1 = expm1(-h)
/ -h - 1 ... (see _rhos).  The hand-off between backbones is the DDIM branch's: after the step at t, `if t < 1000 -
t_switch: model = late`.

Coefficients are fp64 Python floats from the fp32 schedule.  x keeps its dtype: an fp64 x_T gives an fp64 run."""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle import uvit_oracle as O


def _lambda(abar: float) -> float:
    return math.log(math.sqrt(abar)) - math.log(math.sqrt(1 - abar))


def _rhos(rks: list, h: float) -> list:
    """UniPC's bh2 coefficients for the nodes rks (the last one is 1: the new evaluation): solve R rho = b with
    R[i] = rks ** i, b[i] = h_phi_k * i! ... / B(h), hh = -h (data prediction)."""
    hh = -h
    bh = math.expm1(hh)
    h_phi_k = math.expm1(hh) / hh - 1
    fact, R, b = 1, [], []
    for i in range(1, len(rks) + 1):
        R.append([rk ** (i - 1) for rk in rks])
        b.append(h_phi_k * fact / bh)
        fact *= i + 1
        h_phi_k = h_phi_k / hh - 1 / fact
    if len(rks) == 1:
        return [0.5]  # UniPC's order-1 corrector
    return [float(v) for v in np.linalg.solve(np.array(R), np.array(b))]


def sample_unipc(early, late, t_switch, x_T: torch.Tensor, n: int, y=None, rule: str = "predict_noise",
                 trace: dict | None = None, use_corrector: bool = True) -> torch.Tensor:
    """UniPC over the n-point DDIM grid (n - 1 model evaluations); returns x at t = 0.  use_corrector=False gives the
    predictor alone (UniP-2)."""
    if rule not in ("predict_noise", "predict_original"):
        raise ValueError(f"UniPC needs a noise or data prediction, not {rule!r}")
    ab = [float(v) for v in O.ddpm_schedule()["alphas_bar"]]
    al = [math.sqrt(v) for v in ab]
    sg = [math.sqrt(1 - v) for v in ab]
    lam = [_lambda(v) for v in ab]
    ts = O.ddim_timesteps(n)
    evals = len(ts) - 1
    order = [1 if k == 0 or k == evals - 1 else 2 for k in range(evals)]
    x, model, xc, Ds = x_T, early, None, []
    for k in range(evals):
        t, s = ts[k], ts[k + 1]
        with torch.no_grad():
            out = model(x, t * torch.ones(x.shape[0], device=x.device), y)
        d = (x - sg[t] * out) / al[t] if rule == "predict_noise" else out
        if trace is not None:
            trace.setdefault("t", []).append(t)
            trace.setdefault("late", []).append(model is late)
            trace.setdefault("out", []).append(out)
        if k == 0 or not use_corrector:
            xc = x
        else:  # UniC from xc_{k-1} at t_{k-1} to t, order p_{k-1}
            tp, p = ts[k - 1], order[k - 1]
            h = lam[t] - lam[tp]
            bh = math.expm1(-h)
            rks = [(lam[ts[k - 1 - i]] - lam[tp]) / h for i in range(1, p)] + [1.0]
            rho = _rhos(rks, h)
            corr = sum(rho[i] * (Ds[-1 - (i + 1)] - Ds[-1]) / rks[i] for i in range(p - 1))
            xc = (sg[t] / sg[tp]) * xc - al[t] * math.expm1(-h) * Ds[-1] - al[t] * bh * (corr + rho[-1] * (d - Ds[-1]))
        Ds.append(d)
        # UniP from xc_k at t to s, order p_k
        h = lam[s] - lam[t]
        bh = math.expm1(-h)
        x = (sg[s] / sg[t]) * xc - al[s] * math.expm1(-h) * d
        if order[k] == 2:
            r = (lam[ts[k - 1]] - lam[t]) / h
            x = x - al[s] * bh * 0.5 * (Ds[-2] - d) / r
        if late is not None and t < 1000 - t_switch:
            model = late
    return x
