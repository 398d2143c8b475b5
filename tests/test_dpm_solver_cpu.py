"""CPU tests of DPM-Solver++(2M): the coefficient table (ddpm.dpm_solver_coefficients) against the textbook oracle
(oracle/dpm_solver_oracle.py), the oracle's first-order form against the DDIM oracle, its convergence on an analytic
model, the `--dpm_solver_steps` flag, the argument checks of get_samples and the C ABI.

Convergence (test_convergence_on_a_gaussian): data N(mu, s^2 I) in 64 dimensions, s = 2, fp64.  The exact eps is
eps*(x, t) = sigma_t (x - alpha_t mu) / (alpha_t^2 s^2 + sigma_t^2), and the probability-flow ODE maps x_T to
x_0 = alpha_0 mu + sqrt(alpha_0^2 s^2 + sigma_0^2) (x_T - alpha_T mu) / sqrt(alpha_T^2 s^2 + sigma_T^2).
Measured rel-L2 of x_0 (n grid points, n - 1 model evaluations):
    n        10      16      20      25      32      50      64      100     128
    2M       9.8e-3  5.5e-2  3.4e-2  2.1e-2  1.2e-2  4.5e-3  2.7e-3  1.0e-3  6.0e-4
    DDIM     1.3e-1  8.2e-2  6.5e-2  5.2e-2  4.1e-2  2.6e-2  2.0e-2  1.3e-2  1.0e-2
Fitted order over n >= 16 (against n - 1): 2M 2.12, DDIM 0.98.
The jump from n = 10 to n = 16 is the final step: from n - 1 = 15 evaluations on it is second order, and on this
integer, uniform-in-t grid its r = h_prev / h is about 0.23, so the extrapolation weight w1 is about -2.2.  With
narrower data (s <= 1) that step dominates the error and 2M is above DDIM at n = 16..25 (s = 1: 1.5e-1 against
9.9e-2 at n = 16; with a first-order final step 6.4e-3).  The rule is the common implementations' lower_order_final
and is kept; DESIGN.md section 3c records the finding."""
import math

import numpy as np
import pytest
import torch

from duodiff_b200 import _lib, sampler
from duodiff_b200.configs import CONFIGS
from duodiff_b200.ddpm import ddim_timesteps, dpm_solver_coefficients
from oracle import dpm_solver_oracle as P
from oracle import uvit_oracle as O

torch.set_num_threads(4)


# ------------------------------------------------------------------------------------------------ table
@pytest.mark.parametrize("n", [2, 10, 15, 16, 20, 50])
@pytest.mark.parametrize("rule", ["predict_noise", "predict_original"])
def test_table_matches_the_oracle(n, rule):
    table, mode = dpm_solver_coefficients(n, rule)
    assert mode == 3 and table.dtype == torch.float32 and tuple(table.shape) == (1000, 8)
    steps = P.steps(n)
    on_grid = {st["t"] for st in steps}
    for st in steps:
        if rule == "predict_noise":
            a, b = 1 / st["alpha_t"], -st["sigma_t"] / st["alpha_t"]
        else:
            a, b = 0.0, 1.0
        if st["order"] == 2:
            w0, w1 = 1 + 1 / (2 * st["r"]), -1 / (2 * st["r"])
        else:
            w0, w1 = 1.0, 0.0
        want = [a, b, st["sigma_s"] / st["sigma_t"], -st["alpha_s"] * math.expm1(-st["h"]), w0, w1, st["order"], 0.0]
        got = table[st["t"]].double().tolist()
        for j, (g, w) in enumerate(zip(got, want)):
            assert g == float(np.float32(w)), (n, rule, st["t"], j, g, w)  # fp64 rounded once to fp32
    off = [t for t in range(1000) if t not in on_grid]
    assert torch.equal(table[off], torch.zeros(len(off), 8))
    orders = [st["order"] for st in steps]
    assert orders[0] == 1 and set(orders[1:-1]) <= {2}
    assert orders[-1] == (1 if n - 1 < 15 else 2) or n == 2
    assert [st["t"] for st in steps] == ddim_timesteps(n)[:-1]


def test_table_rejects_bad_arguments():
    with pytest.raises(ValueError, match="predict_previous"):
        dpm_solver_coefficients(20, "predict_previous")
    for bad in (0, 1):
        with pytest.raises(ValueError, match="at least 2"):
            dpm_solver_coefficients(bad)


# ------------------------------------------------------------------------------------------------ oracle
def _nonlinear_eps(x, t, y):
    return torch.tanh(0.7 * x + torch.sin(t / 97.0).view(-1, *([1] * (x.dim() - 1))))


def test_order_one_is_ddim(monkeypatch):
    """DPM-Solver++ with every step first order is DDIM at eta = 0 (the same exponential-integrator step).  Both run
    in fp64: the DDIM oracle's schedule is promoted to fp64 so that its coefficients are not rounded to fp32."""
    fp32 = O.ddpm_schedule
    monkeypatch.setattr(O, "ddpm_schedule", lambda device="cpu": {k: v.double() for k, v in fp32(device).items()})
    g = torch.Generator().manual_seed(3)
    x_T = torch.randn(3, 4, 8, 8, generator=g, dtype=torch.float64)
    zero = lambda t: torch.zeros_like(x_T)  # noqa: E731  (eta = 0: the noise term vanishes)
    for n in (2, 10, 20, 50):
        ref = O.sample_ddim(_nonlinear_eps, None, math.inf, x_T.clone(), zero, n, 0.0)
        got = P.sample_dpm_solver(_nonlinear_eps, None, math.inf, x_T.clone(), n, force_order=1)
        assert float((got - ref).norm() / ref.norm()) <= 1e-10, n


def test_oracle_hands_off_like_ddim():
    early = lambda x, t, y: 0.1 * x  # noqa: E731
    late = lambda x, t, y: 0.2 * x  # noqa: E731
    tr_p, tr_d = {}, {}
    x = torch.randn(1, 3, 4, 4)
    P.sample_dpm_solver(early, late, 300, x, 20, trace=tr_p)
    O.sample_ddim(early, late, 300, x, lambda t: torch.zeros_like(x), 20, 0.0, trace=tr_d)
    assert tr_p["t"] == tr_d["t"] and tr_p["late"] == tr_d["late"] and any(tr_p["late"])


def test_convergence_on_a_gaussian():
    sch = O.ddpm_schedule()["alphas_bar"].double()
    al, sg = sch.sqrt(), (1 - sch).sqrt()
    s = 2.0
    g = torch.Generator().manual_seed(0)
    mu = torch.randn(64, generator=g, dtype=torch.float64)

    def eps(x, t, y):
        a, si = al[int(t[0])], sg[int(t[0])]
        return si * (x - a * mu) / (a * a * s * s + si * si)
    x_T = torch.randn(8, 64, generator=g, dtype=torch.float64)
    exact = al[0] * mu + torch.sqrt(al[0] ** 2 * s * s + sg[0] ** 2) * (x_T - al[999] * mu) / \
        torch.sqrt(al[999] ** 2 * s * s + sg[999] ** 2)
    ns = [10, 16, 20, 25, 32, 50, 64, 100, 128]
    err2, err1 = [], []
    for n in ns:
        for errs, order in ((err2, None), (err1, 1)):
            x0 = P.sample_dpm_solver(eps, None, math.inf, x_T.clone(), n, force_order=order)
            errs.append(float((x0 - exact).norm() / exact.norm()))
    nfe = np.array(ns, dtype=float) - 1
    fit = nfe >= 15
    p2 = -np.polyfit(np.log(nfe[fit]), np.log(np.array(err2)[fit]), 1)[0]
    p1 = -np.polyfit(np.log(nfe[fit]), np.log(np.array(err1)[fit]), 1)[0]
    print(f"2M {['%.1e' % e for e in err2]} order {p2:.2f}; DDIM {['%.1e' % e for e in err1]} order {p1:.2f}")
    assert p2 >= 1.8 and p1 <= 1.3
    assert all(a < b for a, b in zip(err2, err1))


# ------------------------------------------------------------------------------------------------ command line
def _base_argv():
    return ["--checkpoint_path", "a.pth", "--batch_size", "4", "--parametrization", "predict_noise",
            "--output_folder", "o", "--config_path", "c.yaml"]


def test_dpm_solver_steps_flag():
    a = sampler.get_args(_base_argv())
    assert "dpm_solver_steps" not in vars(a)  # unset: the namespace of the reference's flags, nothing more
    assert sorted(vars(a)) == sorted(["seed", "checkpoint_path", "checkpoint_path_late", "batch_size",
                                      "parametrization", "output_folder", "config_path", "config_path_late",
                                      "t_switch", "class_id", "use_ddim", "ddim_steps", "ddim_eta", "timesteps_save"])
    a = sampler.get_args(_base_argv() + ["--dpm_solver_steps", "20"])
    assert a.dpm_solver_steps == 20 and not a.use_ddim
    a = sampler.get_args(_base_argv() + ["--dpm_solver_steps", "20", "--class_id", "1", "--cfg_scale", "1.5",
                                         "--timesteps_save", "100", "900"])
    assert a.dpm_solver_steps == 20 and a.cfg_scale == 1.5 and a.timesteps_save == [100, 900]
    argv = _base_argv()
    argv[argv.index("predict_noise")] = "predict_previous"
    for bad in (_base_argv() + ["--dpm_solver_steps", "20", "--use_ddim"], argv + ["--dpm_solver_steps", "20"],
                _base_argv() + ["--dpm_solver_steps", "1"]):
        with pytest.raises(SystemExit):
            sampler.get_args(bad)


def _small(name):
    import duodiff_b200 as ddb
    return ddb.UViT(**dict(CONFIGS[name], embed_dim=64, num_heads=2, depth=1))


def test_get_samples_rejects_bad_dpm_solver_arguments():
    import duodiff_b200 as ddb
    kw = dict(batch_size=2, seed=0, num_channels=4, sample_height=32, sample_width=32)
    net = _small("imagenet256_3")
    pn = sampler.predict_noise_postprocessing
    with pytest.raises(ValueError, match="use_ddim"):
        sampler.get_samples(net, postprocessing=pn, use_ddim=True, dpm_solver_steps=20, **kw)
    with pytest.raises(ValueError, match="predict_previous"):
        sampler.get_samples(net, postprocessing=sampler.predict_previous_postprocessing, dpm_solver_steps=20, **kw)
    with pytest.raises(ValueError, match="at least 2"):
        sampler.get_samples(net, postprocessing=pn, dpm_solver_steps=1, **kw)
    with pytest.raises(ValueError, match="early exit"):
        sampler.get_samples(ddb.EarlyExitUViT(net, "mlp_probe_per_layer"), postprocessing=pn, dpm_solver_steps=20, **kw)
    assert sampler._dpm_solver_rule([net], "predict_original", False, 20) == ("dpm_solver++", 20, "predict_original")


def test_mode_3_in_the_exported_abi():
    from pathlib import Path

    from duodiff_b200 import _build
    _build.build()
    lib = _lib.load()
    for sym in ("ddb_sampler_create", "ddb_sampler_run_list", "ddb_sampler_run", "ddb_ddpm_step"):
        assert sym in _lib.EXPORTED_SYMBOLS and hasattr(lib, sym)
    header = (Path(__file__).resolve().parents[1] / "include" / "duodiff_b200.h").read_text()
    assert "step_mode 3" in header and "[1000,8]" in header
