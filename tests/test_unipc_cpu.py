"""CPU tests of UniPC (bh2, order 2, data prediction): the coefficient table (ddpm.unipc_coefficients), the folded
table's arithmetic against the structured UniP / UniC oracle (oracle/unipc_oracle.py), convergence on an analytic
Gaussian against DPM-Solver++(2M), the `--unipc_steps` flag, the argument checks of get_samples and the C header.

Convergence (test_convergence_against_dpm_solver): data N(mu, s^2 I) in 64 dimensions, fp64, exact eps and exact
probability-flow map as in test_dpm_solver_cpu.py.  Rel-L2 of x_0 at n grid points (n - 1 model evaluations):
    n                    6       8       11      16      21      26      51
    s = 1    DDIM        2.1e-1  1.5e-1  1.1e-1  7.5e-2  5.7e-2  4.6e-2  2.3e-2
             2M          1.6e-1  8.5e-2  3.2e-2  1.1e-1  6.8e-2  4.5e-2  1.1e-2
             UniP only   1.6e-1  8.5e-2  3.2e-2  4.9e-3  2.0e-3  3.5e-3  2.5e-3
             UniPC       1.5e-1  7.0e-2  2.2e-2  2.7e-3  1.0e-3  1.6e-3  7.1e-4
    s = 0.5  2M          1.8e-1  1.2e-1  7.2e-2  1.2e-1  9.0e-2  6.7e-2  2.1e-2
             UniP only   1.8e-1  1.2e-1  7.2e-2  3.3e-2  1.5e-2  6.7e-3  1.6e-3
             UniPC       1.7e-1  1.2e-1  6.8e-2  3.0e-2  1.4e-2  6.8e-3  4.1e-5
UniPC is below 2M at every n.  From 15 evaluations on most of the gap is 2M's second-order final step (DESIGN.md
section 3c); the corrector's own gain is the ratio of the UniP-only and UniPC rows: 1.1-1.5x at <= 10 evaluations and
1.8-3.5x from 15 on for s = 1.  For s = 0.5 it is smaller and at n = 26 the corrector is 1 % worse."""
import math

import numpy as np
import pytest
import torch

from duodiff_b200 import sampler
from duodiff_b200.configs import CONFIGS
from duodiff_b200.ddpm import _unipc_table64, ddim_timesteps, unipc_coefficients
from oracle import dpm_solver_oracle as P
from oracle import uvit_oracle as O
from oracle import unipc_oracle as U

torch.set_num_threads(4)


# ------------------------------------------------------------------------------------------------ table
@pytest.mark.parametrize("n", [2, 3, 6, 16, 20, 50])
@pytest.mark.parametrize("rule", ["predict_noise", "predict_original"])
def test_table_layout(n, rule):
    table, mode = unipc_coefficients(n, rule)
    assert mode == 4 and table.dtype == torch.float32 and tuple(table.shape) == (1000, 12)
    assert torch.equal(table, _unipc_table64(n, rule).to(torch.float32))
    ts = ddim_timesteps(n)
    steps = ts[:-1]
    pred = [int(table[t, 10]) for t in steps]
    corr = [int(table[t, 9]) for t in steps]
    assert pred == [1] + [2] * (len(steps) - 2) + [1] if len(steps) >= 2 else pred == [1]
    assert corr == [0] + pred[:-1]  # the corrector's order is that of the predictor that produced x
    off = [t for t in range(1000) if t not in steps]
    assert torch.equal(table[off], torch.zeros(len(off), 12))
    assert bool((table[steps, 11] == 0).all())
    first = table[ts[0]]
    assert torch.equal(first[2:6], torch.zeros(4))  # no corrector at the first grid point
    for t in steps:
        if table[t, 9] < 2:
            assert table[t, 5] == 0  # no D2 term below corrector order 2
        if table[t, 10] < 2:
            assert table[t, 8] == 0  # no D1 term in a first-order predictor
    if rule == "predict_original":
        assert bool((table[steps, 0] == 0).all()) and bool((table[steps, 1] == 1).all())


def test_table_of_two_points_is_ddim():
    """n = 2: one first-order step without corrector, the DDIM (eta = 0) step from 999 to 0."""
    table = _unipc_table64(2)
    ab = O.ddpm_schedule()["alphas_bar"].double()
    a, s = ab.sqrt(), (1 - ab).sqrt()
    row = table[999]
    assert row[9] == 0 and row[10] == 1
    # x' = px*x + p0*(x - sigma*eps)/alpha = sqrt(ab_0/ab_999)*x + (s_0 - a_0*s_999/a_999)*eps ... as in DDIM
    cx = row[6] + row[7] * row[0]
    ce = row[7] * row[1]
    assert abs(float(cx - a[0] / a[999])) < 1e-12
    assert abs(float(ce - (s[0] - a[0] * s[999] / a[999]))) < 1e-12


def test_table_rejects_bad_arguments():
    with pytest.raises(ValueError, match="predict_previous"):
        unipc_coefficients(20, "predict_previous")
    for bad in (0, 1):
        with pytest.raises(ValueError, match="at least 2"):
            unipc_coefficients(bad)


# ------------------------------------------------------------------------------------------------ folded == oracle
def folded_loop(early, late, t_switch, x_T, n, y=None, rule="predict_noise", table=None):
    """The step kernel's arithmetic over the folded table (fp64 table: no rounding of the coefficients)."""
    table = _unipc_table64(n, rule) if table is None else table
    x, model = x_T, early
    xb = d1 = d2 = None
    for t in ddim_timesteps(n)[:-1]:
        a, b, cx, c0, c1, c2, px, p0, p1, corr, pred, _ = (float(v) for v in table[t])
        out = model(x, t * torch.ones(x.shape[0]), y)  # the oracle's fp32 timestep vector
        d = a * x + b * out
        xc = x
        if corr >= 1:
            xc = cx * xb + c0 * d + c1 * d1
            if corr == 2:
                xc = xc + c2 * d2
        x = px * xc + p0 * d
        if pred == 2:
            x = x + p1 * d1
        xb, d2, d1 = xc, d1 if corr >= 1 else None, d
        if late is not None and t < 1000 - t_switch:
            model = late
    return x


@pytest.mark.parametrize("n", [2, 3, 6, 10, 20, 50])
@pytest.mark.parametrize("rule", ["predict_noise", "predict_original"])
def test_folded_table_equals_the_oracle_on_a_linear_model(n, rule):
    g = torch.Generator().manual_seed(n)
    A = torch.randn(48, 48, generator=g, dtype=torch.float64) / 48 ** 0.5
    c = torch.randn(48, generator=g, dtype=torch.float64)

    def f(x, t, y):
        return x @ A.T * 0.3 + torch.cos(t / 211.0).view(-1, 1) * c

    x_T = torch.randn(5, 48, generator=g, dtype=torch.float64)
    ref = U.sample_unipc(f, None, math.inf, x_T.clone(), n, rule=rule)
    got = folded_loop(f, None, math.inf, x_T.clone(), n, rule=rule)
    assert float((got - ref).norm() / ref.norm()) <= 1e-12, n


def test_folded_table_hands_off_like_the_oracle():
    early = lambda x, t, y: 0.1 * x  # noqa: E731
    late = lambda x, t, y: -0.2 * x + 0.05  # noqa: E731
    x = torch.randn(2, 16, dtype=torch.float64)
    tr = {}
    ref = U.sample_unipc(early, late, 300, x.clone(), 20, trace=tr)
    assert any(tr["late"]) and not all(tr["late"])
    got = folded_loop(early, late, 300, x.clone(), 20)
    assert float((got - ref).norm() / ref.norm()) <= 1e-12
    tr_d = {}
    O.sample_ddim(early, late, 300, x, lambda t: torch.zeros_like(x), 20, 0.0, trace=tr_d)
    assert tr["t"] == tr_d["t"] and tr["late"] == tr_d["late"]


def _gaussian(s):
    sch = O.ddpm_schedule()["alphas_bar"].double()
    al, sg = sch.sqrt(), (1 - sch).sqrt()
    g = torch.Generator().manual_seed(0)
    mu = torch.randn(64, generator=g, dtype=torch.float64)

    def eps(x, t, y):
        a, si = al[int(t[0])], sg[int(t[0])]
        return si * (x - a * mu) / (a * a * s * s + si * si)
    x_T = torch.randn(8, 64, generator=g, dtype=torch.float64)
    exact = al[0] * mu + torch.sqrt(al[0] ** 2 * s * s + sg[0] ** 2) * (x_T - al[999] * mu) / \
        torch.sqrt(al[999] ** 2 * s * s + sg[999] ** 2)
    return eps, x_T, exact


def test_folded_table_equals_the_oracle_on_a_gaussian():
    eps, x_T, _ = _gaussian(1.0)
    for n in (6, 16, 51):
        ref = U.sample_unipc(eps, None, math.inf, x_T.clone(), n)
        got = folded_loop(eps, None, math.inf, x_T.clone(), n)
        assert float((got - ref).norm() / ref.norm()) <= 1e-12, n


def test_oracle_without_corrector_is_the_predictor():
    """UniP alone with a first-order step everywhere is DDIM (eta = 0); the corrector changes the result."""
    eps, x_T, _ = _gaussian(1.0)
    up = U.sample_unipc(eps, None, math.inf, x_T.clone(), 3, use_corrector=False)  # two first-order steps
    ddim = P.sample_dpm_solver(eps, None, math.inf, x_T.clone(), 3, force_order=1)
    assert float((up - ddim).norm() / ddim.norm()) <= 1e-12
    assert not torch.allclose(U.sample_unipc(eps, None, math.inf, x_T.clone(), 3), up)


# ------------------------------------------------------------------------------------------------ convergence
@pytest.mark.parametrize("s", [1.0, 0.5])
def test_convergence_against_dpm_solver(s):
    eps, x_T, exact = _gaussian(s)
    ns = [6, 8, 11, 16, 21, 26, 51]
    err = {"2M": [], "UniP": [], "UniPC": []}
    for n in ns:
        for name, run in (("2M", lambda: P.sample_dpm_solver(eps, None, math.inf, x_T.clone(), n)),
                          ("UniP", lambda: U.sample_unipc(eps, None, math.inf, x_T.clone(), n, use_corrector=False)),
                          ("UniPC", lambda: U.sample_unipc(eps, None, math.inf, x_T.clone(), n))):
            err[name].append(float((run() - exact).norm() / exact.norm()))
    for name, e in err.items():
        print(f"s = {s} {name:6s}", " ".join(f"{v:.1e}" for v in e))
    assert all(u < d for u, d in zip(err["UniPC"], err["2M"]))
    if s == 1.0:
        assert all(u < p for u, p in zip(err["UniPC"], err["UniP"]))  # the corrector helps at every n


# ------------------------------------------------------------------------------------------------ command line
def _base_argv():
    return ["--checkpoint_path", "a.pth", "--batch_size", "4", "--parametrization", "predict_noise",
            "--output_folder", "o", "--config_path", "c.yaml"]


def test_unipc_steps_flag():
    a = sampler.get_args(_base_argv())
    assert "unipc_steps" not in vars(a)  # unset: the namespace of the reference's flags, nothing more
    a = sampler.get_args(_base_argv() + ["--unipc_steps", "16"])
    assert a.unipc_steps == 16 and not a.use_ddim and "dpm_solver_steps" not in vars(a)
    a = sampler.get_args(_base_argv() + ["--unipc_steps", "16", "--class_id", "1", "--cfg_scale", "1.5",
                                         "--timesteps_save", "100", "900"])
    assert a.unipc_steps == 16 and a.cfg_scale == 1.5 and a.timesteps_save == [100, 900]
    argv = _base_argv()
    argv[argv.index("predict_noise")] = "predict_previous"
    for bad in (_base_argv() + ["--unipc_steps", "16", "--use_ddim"],
                _base_argv() + ["--unipc_steps", "16", "--dpm_solver_steps", "16"],
                argv + ["--unipc_steps", "16"], _base_argv() + ["--unipc_steps", "1"]):
        with pytest.raises(SystemExit):
            sampler.get_args(bad)


def test_get_samples_rejects_bad_unipc_arguments():
    import duodiff_b200 as ddb
    kw = dict(batch_size=2, seed=0, num_channels=4, sample_height=32, sample_width=32)
    net = ddb.UViT(**dict(CONFIGS["imagenet256_3"], embed_dim=64, num_heads=2, depth=1))
    pn = sampler.predict_noise_postprocessing
    with pytest.raises(ValueError, match="use_ddim"):
        sampler.get_samples(net, postprocessing=pn, use_ddim=True, unipc_steps=16, **kw)
    with pytest.raises(ValueError, match="dpm_solver_steps"):
        sampler.get_samples(net, postprocessing=pn, dpm_solver_steps=16, unipc_steps=16, **kw)
    with pytest.raises(ValueError, match="predict_previous"):
        sampler.get_samples(net, postprocessing=sampler.predict_previous_postprocessing, unipc_steps=16, **kw)
    with pytest.raises(ValueError, match="at least 2"):
        sampler.get_samples(net, postprocessing=pn, unipc_steps=1, **kw)
    with pytest.raises(ValueError, match="early exit"):
        sampler.get_samples(ddb.EarlyExitUViT(net, "mlp_probe_per_layer"), postprocessing=pn, unipc_steps=16, **kw)
    assert sampler._unipc_rule([net], "predict_original", False, None, 16) == ("unipc", 16, "predict_original")


def test_header_documents_step_mode_4():
    from pathlib import Path
    header = (Path(__file__).resolve().parents[1] / "include" / "duodiff_b200.h").read_text()
    assert "step_mode 4" in header and "[1000,12]" in header and "unipc_coefficients" in header
