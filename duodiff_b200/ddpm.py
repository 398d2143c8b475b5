"""DDPM schedule + the Python owner of a ``ddb_sampler`` handle (the whole t-loop runs inside the C library)."""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib
from .engine import Engine

import numpy as np

RULES = ("predict_noise", "predict_original", "predict_previous")


def ddim_timesteps(ddim_steps: int) -> list:
    """sampler.py:104 — np.linspace(0, 999, ddim_steps).astype(int)[::-1]."""
    ts = [int(v) for v in np.linspace(0, 999, ddim_steps).astype(int)[::-1]]
    if any(s >= t for t, s in zip(ts[:-1], ts[1:])):
        raise ValueError(f"ddim_steps={ddim_steps}: the strided schedule must be strictly decreasing (sampler.py:106)")
    return ts


def ddim_coefficients(ddim_steps: int, ddim_eta: float):
    """[1000,4] fp32 table {c0, c1, sigma2, d} for the DDIM update (sampler.py:110-120), mode 2 of the step kernel:
        x' = (c0*(x - c1*eps) + d*eps) + sigma2*z,   c0 = sqrt(abar_s/abar_t), c1 = sqrt(1-abar_t),
        d = sqrt(1 - abar_s - sigma2), sigma2 = betas_tilde[t]*eta (the reference adds sigma_t^2 * z), z = 0 if s == 0.
    Rows of timesteps the schedule does not visit stay zero."""
    sch = schedule()
    ab, bt = sch["alphas_bar"], sch["betas_tilde"]
    table = torch.zeros(1000, 4, dtype=torch.float32)
    ts = ddim_timesteps(ddim_steps)
    for t, s in zip(ts[:-1], ts[1:]):
        sigma2 = bt[t] * ddim_eta
        table[t, 0] = torch.sqrt(ab[s] / ab[t])
        table[t, 1] = torch.sqrt(1 - ab[t])
        table[t, 2] = sigma2 if s > 0 else 0.0
        table[t, 3] = torch.sqrt(1 - ab[s] - sigma2)
    return table.contiguous(), 2


def dpm_solver_coefficients(steps: int, parametrization: str = "predict_noise"):
    """[1000,8] fp32 table {a, b, rho, phi, w0, w1, order, 0} of DPM-Solver++(2M), mode 3 of the step kernel, over
    the DDIM grid ddim_timesteps(steps) (steps - 1 model evaluations).  With alpha = sqrt(abar), sigma = sqrt(1 - abar),
    lambda = log(alpha / sigma), the step from t to the next grid point s, h = lambda_s - lambda_t, r = h_prev / h:
        D_t = a*x + b*out            predict_noise: a = 1/alpha_t, b = -sigma_t/alpha_t;  predict_original: a = 0, b = 1
        D   = w0*D_t + w1*D_prev     order 2: w0 = 1 + 1/(2r), w1 = -1/(2r);  order 1: D = D_t (w0 = 1, w1 = 0)
        x'  = rho*x + phi*D          rho = sigma_s/sigma_t, phi = alpha_s * (-expm1(-h));  D_prev <- D_t
    The first step is order 1, and so is the final one when the grid has fewer than 15 model evaluations (the usual
    lower_order_final rule: h of the step to t = 0 is large).  Computed in fp64 from the fp32 schedule, rounded once.
    Rows of timesteps no step starts from have order 0."""
    if parametrization not in ("predict_noise", "predict_original"):
        raise ValueError(f"DPM-Solver++ needs a data or noise prediction, not {parametrization!r}")
    if int(steps) < 2:
        raise ValueError(f"dpm_solver_steps={steps}: the grid needs at least 2 points (one model evaluation)")
    ab = schedule()["alphas_bar"].double()
    alpha, sigma = ab.sqrt(), (1 - ab).sqrt()
    lam = alpha.log() - sigma.log()
    ts = ddim_timesteps(int(steps))
    evals = len(ts) - 1
    table = torch.zeros(1000, 8, dtype=torch.float64)
    for k, (t, s) in enumerate(zip(ts[:-1], ts[1:])):
        h = float(lam[s] - lam[t])
        order = 1 if k == 0 or (k == evals - 1 and evals < 15) else 2
        w0, w1 = 1.0, 0.0
        if order == 2:
            r = float(lam[t] - lam[ts[k - 1]]) / h
            w0, w1 = 1 + 1 / (2 * r), -1 / (2 * r)
        a, b = (0.0, 1.0) if parametrization == "predict_original" else (float(1 / alpha[t]),
                                                                        float(-sigma[t] / alpha[t]))
        table[t] = torch.tensor([a, b, float(sigma[s] / sigma[t]), float(alpha[s]) * -math.expm1(-h), w0, w1, order,
                                 0.0], dtype=torch.float64)
    return table.to(torch.float32).contiguous(), 3


def _unipc_table64(steps: int, parametrization: str = "predict_noise") -> torch.Tensor:
    """The [1000,12] table of unipc_coefficients in fp64, before its single rounding to fp32."""
    if parametrization not in ("predict_noise", "predict_original"):
        raise ValueError(f"UniPC needs a data or noise prediction, not {parametrization!r}")
    if int(steps) < 2:
        raise ValueError(f"unipc_steps={steps}: the grid needs at least 2 points (one model evaluation)")
    ab = schedule()["alphas_bar"].double()
    alpha, sigma = ab.sqrt(), (1 - ab).sqrt()
    lam = [float(v) for v in alpha.log() - sigma.log()]
    alpha, sigma = [float(v) for v in alpha], [float(v) for v in sigma]
    ts = ddim_timesteps(int(steps))
    evals = len(ts) - 1
    order = [1 if k == 0 or k == evals - 1 else 2 for k in range(evals)]  # predictor order (lower_order_final)
    table = torch.zeros(1000, 12, dtype=torch.float64)
    for k in range(evals):
        t, s = ts[k], ts[k + 1]
        a, b = (0.0, 1.0) if parametrization == "predict_original" else (1 / alpha[t], -sigma[t] / alpha[t])
        # corrector from the previous base point to t (order of the predictor that produced x at t)
        cx = c0 = c1 = c2 = 0.0
        corr = order[k - 1] if k > 0 else 0
        if corr:
            h = lam[t] - lam[ts[k - 1]]
            phi = math.expm1(-h)
            bh = phi  # B(h) of the bh2 variant
            al = alpha[t]
            cx = sigma[t] / sigma[ts[k - 1]]
            if corr == 1:
                c0 = -al * bh * 0.5
                c1 = -al * phi + al * bh * 0.5
            else:
                r = (lam[ts[k - 2]] - lam[ts[k - 1]]) / h
                g1 = phi / -h - 1
                g2 = g1 / -h - 0.5
                rho0 = (g1 / bh - 2 * g2 / bh) / (1 - r)  # [[1, 1], [r, 1]] [rho0, rho1] = [g1/B, 2 g2/B]
                rho1 = g1 / bh - rho0
                c0 = -al * bh * rho1
                c1 = -al * phi + al * bh * rho0 / r + al * bh * rho1
                c2 = -al * bh * rho0 / r
        # predictor from the corrected x at t to s
        h = lam[s] - lam[t]
        phi = math.expm1(-h)
        px, p0, p1 = sigma[s] / sigma[t], -alpha[s] * phi, 0.0
        if order[k] == 2:
            r = (lam[ts[k - 1]] - lam[t]) / h
            p0 += alpha[s] * phi / (2 * r)
            p1 = -alpha[s] * phi / (2 * r)
        table[t] = torch.tensor([a, b, cx, c0, c1, c2, px, p0, p1, corr, order[k], 0.0], dtype=torch.float64)
    return table


def unipc_coefficients(steps: int, parametrization: str = "predict_noise"):
    """[1000,12] fp32 table {a, b, cx, c0, c1, c2, px, p0, p1, corrector order, predictor order, 0} of UniPC (Zhao et
    al., 2023: bh2, order 2, data prediction), mode 4 of the step kernel, over the DDIM grid ddim_timesteps(steps)
    (steps - 1 model evaluations).  With alpha = sqrt(abar), sigma = sqrt(1 - abar), lambda = log(alpha / sigma), the
    step that evaluates the model at x_k, t_k computes the data prediction D_k = a*x_k + b*out (predict_noise: a =
    1/alpha, b = -sigma/alpha; predict_original: a = 0, b = 1), then
        corrector  xc_k    = cx*xc_{k-1} + c0*D_k + c1*D_{k-1} + c2*D_{k-2}     (xc_0 = x_0: corrector order 0)
        predictor  x_{k+1} = px*xc_k + p0*D_k + p1*D_{k-1}
    The corrector, UniC, reuses this step's evaluation, so it costs no model call; its order is the order of the
    predictor that produced x_k.  The predictor, UniP, is order 1 on the first and the final step (lower_order_final)
    and 2 otherwise.  The structured form of both is oracle/unipc_oracle.py.  Computed in fp64 from the fp32 schedule,
    rounded once.  Rows of timesteps no step starts from are zero (predictor order 0)."""
    return _unipc_table64(steps, parametrization).to(torch.float32).contiguous(), 4


def _sde_dpm_solver_table64(steps: int, parametrization: str = "predict_noise") -> torch.Tensor:
    """The [1000,8] table of sde_dpm_solver_coefficients in fp64, before its single rounding to fp32."""
    if parametrization not in ("predict_noise", "predict_original"):
        raise ValueError(f"SDE-DPM-Solver++ needs a data or noise prediction, not {parametrization!r}")
    if int(steps) < 2:
        raise ValueError(f"sde_dpm_solver_steps={steps}: the grid needs at least 2 points (one model evaluation)")
    ab = schedule()["alphas_bar"].double()
    alpha, sigma = ab.sqrt(), (1 - ab).sqrt()
    lam = [float(v) for v in alpha.log() - sigma.log()]
    alpha, sigma = [float(v) for v in alpha], [float(v) for v in sigma]
    ts = ddim_timesteps(int(steps))
    evals = len(ts) - 1
    table = torch.zeros(1000, 8, dtype=torch.float64)
    for k, (t, s) in enumerate(zip(ts[:-1], ts[1:])):
        h = lam[s] - lam[t]
        order = 1 if k == 0 or k == evals - 1 else 2
        w0, w1 = 1.0, 0.0
        if order == 2:
            r = (lam[t] - lam[ts[k - 1]]) / h
            w0, w1 = 1 + 1 / (2 * r), -1 / (2 * r)
        a, b = (0.0, 1.0) if parametrization == "predict_original" else (1 / alpha[t], -sigma[t] / alpha[t])
        e2 = -math.expm1(-2 * h)
        vs = sigma[s] * math.sqrt(e2) if s > 0 else 0.0
        table[t] = torch.tensor([a, b, sigma[s] / sigma[t] * math.exp(-h), alpha[s] * e2, w0, w1, order, vs],
                                dtype=torch.float64)
    return table


def sde_dpm_solver_coefficients(steps: int, parametrization: str = "predict_noise"):
    """[1000,8] fp32 table {a, b, rho, phi, w0, w1, order, vs} of SDE-DPM-Solver++(2M) (Lu et al., 2022: the
    second-order multistep solver of the reverse SDE, data prediction), mode 5 of the step kernel, over the DDIM grid
    ddim_timesteps(steps) (steps - 1 model evaluations).  With alpha = sqrt(abar), sigma = sqrt(1 - abar), lambda =
    log(alpha / sigma), the step from t to the next grid point s, h = lambda_s - lambda_t, r = h_prev / h:
        D_t = a*x + b*out            predict_noise: a = 1/alpha_t, b = -sigma_t/alpha_t;  predict_original: a = 0, b = 1
        D   = w0*D_t + w1*D_prev     order 2: w0 = 1 + 1/(2r), w1 = -1/(2r);  order 1: D = D_t (w0 = 1, w1 = 0)
        x'  = rho*x + phi*D + vs*z   rho = (sigma_s/sigma_t) exp(-h), phi = alpha_s (-expm1(-2h)),
                                     vs = sigma_s sqrt(-expm1(-2h)) (0 on the final step, s = 0);  D_prev <- D_t
    z is the draw of the DDPM step at t.  A first-order step is the DDPM posterior (ancestral) step from t to s; for s =
    t - 1 it is the reference's DDPM update.  The first and the final step are order 1, the others order 2.  The
    textbook form is oracle/sde_dpm_solver_oracle.py.  Computed in fp64 from the fp32 schedule, rounded once.  Rows of
    timesteps no step starts from are zero (order 0)."""
    return _sde_dpm_solver_table64(steps, parametrization).to(torch.float32).contiguous(), 5


def schedule() -> dict:
    """The five schedule vectors, built with the reference's own torch calls (sampler.py:40-44) on the host so the
    coefficient table is bit-identical to a CPU run of the reference."""
    betas = torch.linspace(1e-4, 0.02, 1000)
    alphas = 1 - betas
    alphas_bar = torch.cumprod(alphas, dim=0)
    alphas_bar_previous = torch.cat([torch.tensor([1.0]), alphas_bar[:-1]])
    betas_tilde = betas * (1 - alphas_bar_previous) / (1 - alphas_bar)
    return dict(betas=betas, alphas=alphas, alphas_bar=alphas_bar, alphas_bar_previous=alphas_bar_previous,
                betas_tilde=betas_tilde)


def step_coefficients(rule: str = "predict_noise", variance: str = "beta_tilde"):
    """[1000,4] fp32 table {c0, c1, sigma, 0} and the kernel's evaluation mode for a post-processing rule.

    predict_noise    (sampler.py:47-56):  mode 0  x' = c0*(x - c1*eps) + sigma*z, c0 = sqrt(1/a), c1 = (1-a)/sqrt(1-abar)
    predict_original (sampler.py:59-72):  mode 1  x' = (c1*out + c0*x) + sigma*z
    predict_previous (sampler.py:75-79):  mode 1  with c0 = 0, c1 = 1
    variance: 'beta_tilde' (sampler.py:50, eesampler.py:76) or 'beta' (ddpm_core.py:56-79 default)."""
    s = schedule()
    var = s["betas_tilde"] if variance == "beta_tilde" else s["betas"]
    sigma = torch.sqrt(var)
    if rule == "predict_noise":
        c0 = torch.sqrt(1 / s["alphas"])
        c1 = (1 - s["alphas"]) / torch.sqrt(1 - s["alphas_bar"])
        mode = 0
    elif rule == "predict_original":
        c1 = torch.sqrt(s["alphas_bar_previous"]) * s["betas"] / (1 - s["alphas_bar"])
        c0 = torch.sqrt(s["alphas"]) * (1 - s["alphas_bar_previous"]) / (1 - s["alphas_bar"])
        mode = 1
    elif rule == "predict_previous":
        c0, c1, mode = torch.zeros(1000), torch.ones(1000), 1
    else:
        raise ValueError(f"unknown parametrization {rule!r}; expected one of {RULES}")
    table = torch.stack([c0, c1, sigma, torch.zeros(1000)], dim=1).to(torch.float32).contiguous()
    return table, mode


def switch_step(t_switch) -> int:
    """sampler.py:135-136: the swap happens after the step at t == 1000 - t_switch, i.e. `early` runs t >= 1000 -
    t_switch.  The equality can only trigger for integral 1 <= t_switch <= 1000; otherwise the early model runs
    the whole trajectory (the reference default t_switch=inf)."""
    try:
        ts = float(t_switch)
    except (TypeError, ValueError):
        return -1
    if ts != ts or ts in (float("inf"), float("-inf")) or ts != int(ts):
        return -1
    ts = int(ts)
    return 1000 - ts if 1 <= ts <= 1000 else -1


_SAMPLER_CACHE: "dict[tuple, Sampler]" = {}


def cached_sampler(early: Engine, late: "Engine | None", t_switch, batch: int, rule: str = "predict_noise",
                   variance: str = "beta_tilde", ee_threshold: "float | None" = None, ee_mode: int = 0,
                   guidance: "tuple | None" = None) -> "Sampler":
    """Sampler for this (models, batch, rule, guidance): its buffers and captured CUDA graphs are reused across
    get_samples() calls (the graphs read t, the seed and x from sampler-owned device memory, so they do not depend on
    the call)."""
    key = (early.handle.value, late.handle.value if late is not None else None, switch_step(t_switch), batch, rule,
           variance, ee_threshold, ee_mode)
    if guidance is not None:
        key += (("guidance", float(guidance[0]), int(guidance[1])),)
    smp = _SAMPLER_CACHE.get(key)
    if smp is None:
        while len(_SAMPLER_CACHE) >= 4:  # bounded: each entry owns a few x-sized device buffers and two graphs
            _SAMPLER_CACHE.pop(next(iter(_SAMPLER_CACHE)))
        smp = _SAMPLER_CACHE[key] = Sampler(early, late, t_switch, batch, rule, variance, ee_threshold, ee_mode,
                                            guidance=guidance)
    return smp


class Sampler:
    """get_samples()' inner loop (sampler.py:128-139 / eesampler.py:57-82) as one C call."""

    def __init__(self, early: Engine, late: Engine | None, t_switch, batch: int, rule: str = "predict_noise",
                 variance: str = "beta_tilde", ee_threshold: float | None = None, ee_mode: int = 0,
                 guidance: "tuple | None" = None):
        """guidance: (scale, null_label) for classifier-free guidance (ddb_sampler_set_guidance): each step runs the
        backbones on 2 * batch rows, so both engines need max_batch >= 2 * batch; runs then need labels y."""
        self.lib = _lib.load()
        self.early, self.late, self.batch = early, late, batch
        if isinstance(rule, tuple) and rule[0] == "ddim":  # ("ddim", ddim_steps, ddim_eta)
            table, mode = ddim_coefficients(int(rule[1]), float(rule[2]))
        elif isinstance(rule, tuple) and rule[0] == "dpm_solver++":  # ("dpm_solver++", steps, parametrization)
            table, mode = dpm_solver_coefficients(int(rule[1]), rule[2])
        elif isinstance(rule, tuple) and rule[0] == "unipc":  # ("unipc", steps, parametrization)
            table, mode = unipc_coefficients(int(rule[1]), rule[2])
        elif isinstance(rule, tuple) and rule[0] == "sde-dpm_solver++":  # ("sde-dpm_solver++", steps, parametrization)
            table, mode = sde_dpm_solver_coefficients(int(rule[1]), rule[2])
        else:
            table, mode = step_coefficients(rule, variance)
        self.coef = table
        self.device = early.device
        if late is not None and late.device != early.device:
            raise _lib.DuoDiffError(f"early model on {early.device}, late model on {late.device}")
        handle = C.c_void_p()
        # early exit is switched by ee_mode (-1 = off), never by the sign of the threshold: a negative threshold is a
        # legal value of eesampler.py's --threshold (every sample then takes layer 0's head)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_sampler_create(
                early.handle, late.handle if late is not None else None,
                switch_step(t_switch) if late is not None else -1, batch, table.data_ptr(), mode,
                0.0 if ee_threshold is None else float(ee_threshold), -1 if ee_threshold is None else int(ee_mode),
                C.byref(handle)))
        self.handle = handle
        if guidance is not None:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.ddb_sampler_set_guidance(handle, float(guidance[0]), int(guidance[1])))

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            try:
                with torch.cuda.device(self.device):
                    self.lib.ddb_sampler_destroy(h)
            except (AttributeError, TypeError):  # interpreter shutdown: torch is already torn down
                pass
            self.handle = None

    def set_noise_offset(self, first_row: int) -> None:
        """This shard holds rows [first_row, first_row + batch) of a global batch: the in-kernel Philox noise is keyed
        by the GLOBAL element index, so the shards together draw exactly the single-process noise."""
        _lib.check(self.lib.ddb_sampler_set_noise_offset(self.handle, int(first_row)))

    def _check_xy(self, x, y, noise):
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.shape[0] == self.batch
        if x.device != self.device:
            raise _lib.DuoDiffError(f"x is on {x.device} but the sampler's models live on {self.device}")
        if noise is not None:
            assert noise.is_cuda and noise.dtype == torch.float32 and noise.is_contiguous()
            assert noise.shape[0] == 1000 and noise[0].numel() == x.numel()
        if y is not None:
            y = self.early.check_labels(y, self.batch)
            if self.late is not None:
                y = self.late.check_labels(y, self.batch)
        return y

    def profile_step(self, x, t: int, late: bool, y=None) -> dict:
        """Per-kernel-category device time of one eager sampling step as the sampler runs it."""
        y = self._check_xy(x, y, None)
        n = len(Engine.PROF_CATEGORIES)
        ms, cnt = (C.c_float * n)(), (C.c_int32 * n)()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_sampler_profile_step(self.handle, x.data_ptr(), _lib.ptr(y), int(t), int(bool(late)),
                                                         ms, cnt, _lib.current_stream_ptr()))
        return {k: dict(ms=float(ms[i]), launches=int(cnt[i])) for i, k in enumerate(Engine.PROF_CATEGORIES)}

    def run(self, x, y=None, noise=None, seed: int = 0, t_first: int = 999, t_last: int = 0, eps_trace=None,
            x_trace=None, exit_log=None, score_log=None, use_graph: bool = True):
        """In place on x [B,C,H,W] f32 cuda.  noise: None (device Philox) or [1000, *x.shape] f32 cuda indexed by t."""
        y = self._check_xy(x, y, noise)
        graph = bool(use_graph) and eps_trace is None and x_trace is None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_sampler_run(
                self.handle, x.data_ptr(), _lib.ptr(y), _lib.ptr(noise), int(seed) & (2**64 - 1), t_first, t_last,
                _lib.ptr(eps_trace), _lib.ptr(x_trace), _lib.ptr(exit_log), _lib.ptr(score_log), int(graph),
                _lib.current_stream_ptr()))
        return x

    def run_list(self, x, t_list, late_flags, y=None, noise=None, seed: int = 0, eps_trace=None, x_trace=None,
                 exit_log=None, score_log=None, use_graph: bool = True):
        """The same loop over an explicit timestep list (DDIM): model at t_list[k] (late backbone if late_flags[k]),
        then the sampler's update with the coefficients of t_list[k].  exit_log / score_log as in run(): only the rows
        of the timesteps in t_list are written."""
        y = self._check_xy(x, y, noise)
        n = len(t_list)
        assert n == len(late_flags)
        ts = (C.c_int32 * n)(*[int(t) for t in t_list])
        lf = (C.c_uint8 * n)(*[1 if f else 0 for f in late_flags])
        for log, dtype, cols in ((exit_log, torch.int32, self.batch), (score_log, torch.float32, self.early.depth)):
            if log is not None:
                assert log.is_cuda and log.dtype == dtype and log.is_contiguous() and tuple(log.shape) == (1000, cols)
        graph = bool(use_graph) and eps_trace is None and x_trace is None
        args = (self.handle, x.data_ptr(), _lib.ptr(y), _lib.ptr(noise), int(seed) & (2**64 - 1), ts, lf, n,
                _lib.ptr(eps_trace), _lib.ptr(x_trace))
        with torch.cuda.device(self.device):
            if exit_log is None and score_log is None:
                _lib.check(self.lib.ddb_sampler_run_list(*args, int(graph), _lib.current_stream_ptr()))
            else:
                _lib.check(self.lib.ddb_sampler_run_list_logs(*args, _lib.ptr(exit_log), _lib.ptr(score_log),
                                                              int(graph), _lib.current_stream_ptr()))
        return x

    def finalize(self, x):
        """(x + 1) / 2, 'b c h w -> b h w c' (sampler.py:145-146)."""
        B, Cc, H, W = x.shape
        out = torch.empty(B, H, W, Cc, device=x.device, dtype=torch.float32)
        with torch.cuda.device(x.device):
            _lib.check(self.lib.ddb_finalize_nhwc(x.data_ptr(), out.data_ptr(), B, Cc, H, W,
                                                  _lib.current_stream_ptr()))
        return out
