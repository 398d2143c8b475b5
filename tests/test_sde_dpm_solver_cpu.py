"""CPU tests of SDE-DPM-Solver++(2M): the coefficient table (ddpm.sde_dpm_solver_coefficients) against the textbook
oracle (oracle/sde_dpm_solver_oracle.py), the first-order step against the DDPM posterior step and the reference's
DDPM update, the distribution error on Gaussian data, the `--sde_dpm_solver_steps` flag, the argument checks of
get_samples and the C header.

Gaussian data (test_gaussian_distribution_error): data N(0, v), fp64, exact data prediction D(x_t) = alpha_t v /
(alpha_t^2 v + sigma_t^2) x_t, x_T ~ N(0, alpha_999^2 v + sigma_999^2).  Every step is linear in x_T and the z's, so
the oracle runs on coefficient vectors over (x_T, z_1, ...) and the output std is their norm.  The error is |std_out -
std_true| / std_true, std_true^2 = alpha_0^2 v + sigma_0^2: the output is Gaussian, so this is its whole distribution
error (W2 per dimension over std_true).  n grid points, n - 1 model evaluations:
    n                                     6       11      16      21      26      51      101
    v = 1     first order (DDIM eta = 1)  3.99e-1 2.60e-1 1.95e-1 1.57e-1 1.32e-1 7.40e-2 4.00e-2
              2M-SDE                      3.28e-1 5.37e-2 1.80e-2 3.49e-2 3.57e-2 1.90e-2 6.70e-3
    v = 0.25  first order                 5.03e-1 3.33e-1 2.61e-1 2.17e-1 1.86e-1 1.12e-1 6.34e-2
              2M-SDE                      4.89e-1 2.23e-1 9.17e-2 2.66e-2 5.10e-3 3.02e-2 1.59e-2
2M-SDE (first-order final step) is below the first-order sampler at every n.  A second-order final step would give
5.29e-1, 5.64e-1, 4.14e-1, 2.90e-1, 2.09e-1, 6.10e-2, 1.52e-2 for v = 1: worse than first order on most grids (the
r ~ 0.23 final step of DESIGN.md section 3c), so the table's final step is first order on every grid."""
import math

import pytest
import torch

from duodiff_b200 import sampler
from duodiff_b200.configs import CONFIGS
from duodiff_b200.ddpm import _sde_dpm_solver_table64, ddim_timesteps, sde_dpm_solver_coefficients
from oracle import sde_dpm_solver_oracle as S
from oracle import uvit_oracle as O

torch.set_num_threads(4)


def _abar64():
    return [float(v) for v in O.ddpm_schedule()["alphas_bar"]]


# ------------------------------------------------------------------------------------------------ table
@pytest.mark.parametrize("n", [2, 3, 6, 16, 20, 50])
@pytest.mark.parametrize("rule", ["predict_noise", "predict_original"])
def test_table_layout(n, rule):
    table, mode = sde_dpm_solver_coefficients(n, rule)
    assert mode == 5 and table.dtype == torch.float32 and tuple(table.shape) == (1000, 8)
    assert torch.equal(table, _sde_dpm_solver_table64(n, rule).to(torch.float32))
    ts = ddim_timesteps(n)
    steps = ts[:-1]
    order = [int(table[t, 6]) for t in steps]
    assert order == ([1] if len(steps) == 1 else [1] + [2] * (len(steps) - 2) + [1])
    off = [t for t in range(1000) if t not in steps]
    assert torch.equal(table[off], torch.zeros(len(off), 8))
    assert table[steps[-1], 7] == 0  # no noise on the final step (s = 0)
    assert bool((table[steps[:-1], 7] > 0).all())
    for t in steps:
        if table[t, 6] == 1:
            assert table[t, 4] == 1 and table[t, 5] == 0
    if rule == "predict_original":
        assert bool((table[steps, 0] == 0).all()) and bool((table[steps, 1] == 1).all())


def test_table_rejects_bad_arguments():
    with pytest.raises(ValueError, match="predict_previous"):
        sde_dpm_solver_coefficients(20, "predict_previous")
    for bad in (0, 1):
        with pytest.raises(ValueError, match="at least 2"):
            sde_dpm_solver_coefficients(bad)


# ------------------------------------------------------------------------------------------------ table == oracle
def folded_loop(early, late, t_switch, x_T, n, noise, y=None, rule="predict_noise", table=None):
    """The step kernel's arithmetic over the table (fp64 table: no rounding of the coefficients)."""
    table = _sde_dpm_solver_table64(n, rule) if table is None else table
    x, model, d_prev = x_T, early, None
    for t in ddim_timesteps(n)[:-1]:
        a, b, rho, phi, w0, w1, order, vs = (float(v) for v in table[t])
        out = model(x, t * torch.ones(x.shape[0]), y)
        dt = a * x + b * out
        d = w0 * dt + w1 * d_prev if order == 2 else dt
        x = rho * x + phi * d
        if vs != 0:
            x = x + vs * noise[t]
        d_prev = dt
        if late is not None and t < 1000 - t_switch:
            model = late
    return x


@pytest.mark.parametrize("n", [2, 3, 6, 10, 20, 50])
@pytest.mark.parametrize("rule", ["predict_noise", "predict_original"])
def test_table_equals_the_oracle_on_a_linear_model(n, rule):
    g = torch.Generator().manual_seed(n)
    A = torch.randn(48, 48, generator=g, dtype=torch.float64) / 48 ** 0.5
    c = torch.randn(48, generator=g, dtype=torch.float64)

    def f(x, t, y):
        return x @ A.T * 0.3 + torch.cos(t / 211.0).view(-1, 1) * c

    x_T = torch.randn(5, 48, generator=g, dtype=torch.float64)
    noise = torch.randn(1000, 5, 48, generator=g, dtype=torch.float64)
    ref = S.sample_sde_dpm_solver(f, None, math.inf, x_T.clone(), n, noise, rule=rule)
    got = folded_loop(f, None, math.inf, x_T.clone(), n, noise, rule=rule)
    assert float((got - ref).norm() / ref.norm()) <= 1e-12, n


def test_table_hands_off_like_the_oracle():
    early = lambda x, t, y: 0.1 * x  # noqa: E731
    late = lambda x, t, y: -0.2 * x + 0.05  # noqa: E731
    x = torch.randn(2, 16, dtype=torch.float64)
    noise = torch.randn(1000, 2, 16, dtype=torch.float64)
    tr = {}
    ref = S.sample_sde_dpm_solver(early, late, 300, x.clone(), 20, noise, trace=tr)
    assert any(tr["late"]) and not all(tr["late"])
    got = folded_loop(early, late, 300, x.clone(), 20, noise)
    assert float((got - ref).norm() / ref.norm()) <= 1e-12
    tr_d = {}
    O.sample_ddim(early, late, 300, x, lambda t: torch.zeros_like(x), 20, 0.0, trace=tr_d)
    assert tr["t"] == tr_d["t"] and tr["late"] == tr_d["late"]


# ------------------------------------------------------------------------------------------------ first order == DDPM
@pytest.mark.parametrize("n", [11, 51])
def test_first_order_step_is_the_ddpm_posterior_step(n):
    """x_s = mean + std z of q(x_s | x_t, x0) with x0 the data prediction, computed directly from abar."""
    ab = _abar64()
    g = torch.Generator().manual_seed(n)
    for st in S.steps(n, all_first_order=True):
        t, s = st["t"], st["s"]
        x, eps, z = (torch.randn(64, generator=g, dtype=torch.float64) for _ in range(3))
        got, _ = S.step(st, x, eps, None, z)
        x0 = (x - math.sqrt(1 - ab[t]) * eps) / math.sqrt(ab[t])
        beta = 1 - ab[t] / ab[s]
        mean = math.sqrt(ab[s]) * beta / (1 - ab[t]) * x0 + math.sqrt(ab[t] / ab[s]) * (1 - ab[s]) / (1 - ab[t]) * x
        want = mean + (math.sqrt((1 - ab[s]) / (1 - ab[t]) * beta) * z if s > 0 else 0)
        assert float((got - want).abs().max()) <= 1e-10, (n, t)


def test_first_order_step_on_every_timestep_is_the_reference_ddpm_update():
    """On the 1000-point grid s = t - 1: 1/sqrt(alpha_t) (x - beta_t / sqrt(1 - abar_t) eps) + sqrt(beta~_t) z, the
    formula of step_coefficients("predict_noise"), in fp64 from the schedule (alpha_t = abar_t / abar_{t-1})."""
    ab = _abar64()
    g = torch.Generator().manual_seed(3)
    checked = 0
    for st in S.steps(1000, all_first_order=True):
        t, s = st["t"], st["s"]
        assert s == t - 1
        if s == 0:
            continue
        x, eps, z = (torch.randn(32, generator=g, dtype=torch.float64) for _ in range(3))
        got, _ = S.step(st, x, eps, None, z)
        alpha = ab[t] / ab[t - 1]
        beta = 1 - alpha
        beta_tilde = beta * (1 - ab[t - 1]) / (1 - ab[t])
        want = 1 / math.sqrt(alpha) * (x - beta / math.sqrt(1 - ab[t]) * eps) + math.sqrt(beta_tilde) * z
        assert float((got - want).abs().max()) <= 1e-10, t
        checked += 1
    assert checked == 998


# ------------------------------------------------------------------------------------------------ Gaussian data
def _gaussian_error(n, v, all_first_order):
    ab = _abar64()
    al, sg = [math.sqrt(a) for a in ab], [math.sqrt(1 - a) for a in ab]
    ts = ddim_timesteps(n)
    basis = torch.eye(len(ts), dtype=torch.float64)  # x = coefficients over (x_T, z of the step at ts[0], ...)
    col = {t: basis[k + 1:k + 2] for k, t in enumerate(ts[:-1])}

    def data(x, t, y):  # the exact data prediction (predict_original)
        tt = int(t[0])
        return al[tt] * v / (al[tt] ** 2 * v + sg[tt] ** 2) * x
    x_T = math.sqrt(al[999] ** 2 * v + sg[999] ** 2) * basis[:1]
    x = S.sample_sde_dpm_solver(data, None, math.inf, x_T, n, lambda t: col[t], rule="predict_original",
                                all_first_order=all_first_order)
    true = math.sqrt(al[0] ** 2 * v + sg[0] ** 2)
    return abs(float(x.norm()) - true) / true


GAUSSIAN = {  # (v, all_first_order): errors at n = 6, 11, 16, 21, 26, 51, 101
    (1.0, True): [3.99e-1, 2.60e-1, 1.95e-1, 1.57e-1, 1.32e-1, 7.40e-2, 4.00e-2],
    (1.0, False): [3.28e-1, 5.37e-2, 1.80e-2, 3.49e-2, 3.57e-2, 1.90e-2, 6.70e-3],
    (0.25, True): [5.03e-1, 3.33e-1, 2.61e-1, 2.17e-1, 1.86e-1, 1.12e-1, 6.34e-2],
    (0.25, False): [4.89e-1, 2.23e-1, 9.17e-2, 2.66e-2, 5.10e-3, 3.02e-2, 1.59e-2],
}


@pytest.mark.parametrize("v", [1.0, 0.25])
def test_gaussian_distribution_error(v):
    ns = [6, 11, 16, 21, 26, 51, 101]
    err = {f: [_gaussian_error(n, v, f) for n in ns] for f in (True, False)}
    for f, name in ((True, "first order"), (False, "2M-SDE")):
        print(f"v = {v} {name:12s}", " ".join(f"{e:.2e}" for e in err[f]))
        for n, got, want in zip(ns, err[f], GAUSSIAN[(v, f)]):
            # to three digits: within one unit of the third (0.25947 was first rounded to 0.2595, then to 2.60e-1)
            assert abs(got - want) <= 10 ** (math.floor(math.log10(want)) - 2), (v, name, n, got, want)
    assert all(m < o for m, o in zip(err[False], err[True]))


# ------------------------------------------------------------------------------------------------ command line
def _base_argv():
    return ["--checkpoint_path", "a.pth", "--batch_size", "4", "--parametrization", "predict_noise",
            "--output_folder", "o", "--config_path", "c.yaml"]


def test_sde_dpm_solver_steps_flag():
    a = sampler.get_args(_base_argv())
    assert "sde_dpm_solver_steps" not in vars(a)  # unset: the namespace of the reference's flags, nothing more
    a = sampler.get_args(_base_argv() + ["--sde_dpm_solver_steps", "16"])
    assert a.sde_dpm_solver_steps == 16 and not a.use_ddim
    assert "dpm_solver_steps" not in vars(a) and "unipc_steps" not in vars(a)
    a = sampler.get_args(_base_argv() + ["--sde_dpm_solver_steps", "16", "--class_id", "1", "--cfg_scale", "1.5",
                                         "--timesteps_save", "100", "900"])
    assert a.sde_dpm_solver_steps == 16 and a.cfg_scale == 1.5 and a.timesteps_save == [100, 900]
    argv = _base_argv()
    argv[argv.index("predict_noise")] = "predict_previous"
    for bad in (_base_argv() + ["--sde_dpm_solver_steps", "16", "--use_ddim"],
                _base_argv() + ["--sde_dpm_solver_steps", "16", "--dpm_solver_steps", "16"],
                _base_argv() + ["--sde_dpm_solver_steps", "16", "--unipc_steps", "16"],
                argv + ["--sde_dpm_solver_steps", "16"], _base_argv() + ["--sde_dpm_solver_steps", "1"]):
        with pytest.raises(SystemExit):
            sampler.get_args(bad)


def test_get_samples_rejects_bad_sde_dpm_solver_arguments():
    import duodiff_b200 as ddb
    kw = dict(batch_size=2, seed=0, num_channels=4, sample_height=32, sample_width=32)
    net = ddb.UViT(**dict(CONFIGS["imagenet256_3"], embed_dim=64, num_heads=2, depth=1))
    pn = sampler.predict_noise_postprocessing
    with pytest.raises(ValueError, match="use_ddim"):
        sampler.get_samples(net, postprocessing=pn, use_ddim=True, sde_dpm_solver_steps=16, **kw)
    with pytest.raises(ValueError, match="dpm_solver_steps"):
        sampler.get_samples(net, postprocessing=pn, dpm_solver_steps=16, sde_dpm_solver_steps=16, **kw)
    with pytest.raises(ValueError, match="unipc_steps"):
        sampler.get_samples(net, postprocessing=pn, unipc_steps=16, sde_dpm_solver_steps=16, **kw)
    with pytest.raises(ValueError, match="predict_previous"):
        sampler.get_samples(net, postprocessing=sampler.predict_previous_postprocessing, sde_dpm_solver_steps=16,
                            **kw)
    with pytest.raises(ValueError, match="at least 2"):
        sampler.get_samples(net, postprocessing=pn, sde_dpm_solver_steps=1, **kw)
    with pytest.raises(ValueError, match="early exit"):
        sampler.get_samples(ddb.EarlyExitUViT(net, "mlp_probe_per_layer"), postprocessing=pn,
                            sde_dpm_solver_steps=16, **kw)
    assert sampler._sde_dpm_solver_rule([net], "predict_original", False, None, None, 16) == \
        ("sde-dpm_solver++", 16, "predict_original")


def test_header_documents_step_mode_5():
    from pathlib import Path
    header = (Path(__file__).resolve().parents[1] / "include" / "duodiff_b200.h").read_text()
    assert "step_mode 5" in header and "sde_dpm_solver_coefficients" in header and "mode 5" in header
