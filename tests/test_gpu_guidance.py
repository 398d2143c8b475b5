"""GPU tests of classifier-free guidance (`-m gpu`, B200): the guided step tail (step_tail_kernel<C, W, true>), the
sampler's 2B-row forwards, `get_samples(cfg_scale=...)` and `sampler.py --cfg_scale`.

Guided eps = c + s * (c - u), c / u = rows [0, B) / [B, 2B) of ONE forward on [x ; x] with labels [y ; null].  The
tail rounds each of the three operations on its own, so the composition is checked bit for bit against torch.

Oracle parity (test_free_running_guided_trajectory_matches_the_oracle): reference-init ImageNet-256 depth-3 backbone,
1000 guided DDPM steps at s = 0.4, injected noise, fp32 oracle (oracle/guidance_oracle.py, TF32 off).  Guidance
amplifies the eps error by about (1 + 2s), so the unguided bound for reference-init weights (5e-3, test_gpu_parity.py)
becomes 5e-3 * (1 + 2 * 0.4) = 9e-3.  Measured on a B200: 1.38e-3.  (At reference init the labels move eps little:
the guided and unguided oracle trajectories differ by 5.4e-4, so the bit-exact composition tests above are what
pins the guided arithmetic.)
"""
import os
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import guidance_oracle as G
from oracle import uvit_oracle as O
from tests.helpers import CONFIGS, heat_, rel_l2
from tests.process_tree import run_tree

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
SCALE = 0.4
IMG_REL_L2_GUIDED = 5e-3 * (1 + 2 * SCALE)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda:0")


def _model(name, seed, hot, dev):
    import duodiff_b200 as ddb
    torch.manual_seed(seed)
    net = ddb.UViT(**CONFIGS[name])
    if hot:  # x2 Linear scale: the 17- and 21-block backbones stay finite over a whole trajectory
        heat_(net, seed + 100, scale=2.0)
    return net.eval().to(dev)


def _null(net):
    return net.num_classes - 1


def _guided_eps(net, x, t, y, null, s):
    """The reference composition: one forward on 2B rows, then three separately rounded torch ops."""
    B = x.shape[0]
    out = net(torch.cat([x, x]), torch.full((2 * B,), float(t), device=x.device),
              torch.cat([y, torch.full_like(y, null)]))
    c, u = out[:B], out[B:]
    d = c - u
    m = s * d
    return c + m


def _lib():
    from duodiff_b200 import _lib
    return _lib, _lib.load()


# ------------------------------------------------------------------------------------------------ composition
@pytest.mark.parametrize("pair", [("imagenet64_3", "imagenet64"), ("imagenet256_3", "imagenet256")])
@pytest.mark.parametrize("rule", ["predict_noise", "predict_original", "ddim"])
def test_guided_step_is_the_torch_composition_bit_for_bit(dev, pair, rule):
    """One eager guided step at a time with injected noise, across the DuoDiff hand-off: eps_trace == c + s (c - u)
    and x_trace == ddb_ddpm_step(x, that eps)."""
    lib, L = _lib()
    from duodiff_b200.ddpm import Sampler, ddim_coefficients, step_coefficients
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model(pair[0], 41, True, dev), _model(pair[1], 42, True, dev)
    B, C, H = 3, early.in_chans, early.img_size
    g = torch.Generator(device=dev).manual_seed(5)
    x_T = torch.randn(B, C, H, H, device=dev, generator=g)
    y = torch.randint(0, early.num_classes - 1, (B,), device=dev, generator=g)
    noise = torch.randn(1000, B, C, H, H, device=dev, generator=g)
    null, s = _null(early), 1.75
    if rule == "ddim":
        steps, flags = _ddim_plan(50, True, 300)
        k0 = flags.index(True) - 3
        ts, fl = steps[k0:k0 + 6], flags[k0:k0 + 6]
        table, mode = ddim_coefficients(50, 0.05)
        smp = Sampler(early.engine(2 * B), late.engine(2 * B), 300, B, rule=("ddim", 50, 0.05), guidance=(s, null))
    else:
        ts = list(range(702, 696, -1))
        fl = [t < 700 for t in ts]
        table, mode = step_coefficients(rule)
        smp = Sampler(early.engine(2 * B), late.engine(2 * B), 300, B, rule=rule, guidance=(s, null))
    assert any(fl) and not all(fl)
    coef = table.to(dev)
    n = len(ts)
    eps_tr, x_tr = torch.zeros(n, B, C, H, H, device=dev), torch.zeros(n, B, C, H, H, device=dev)
    x = x_T.clone()
    if rule == "ddim":
        smp.run_list(x, ts, fl, y=y, noise=noise, eps_trace=eps_tr, x_trace=x_tr, use_graph=False)
    else:
        smp.run(x, y=y, noise=noise, t_first=ts[0], t_last=ts[-1], eps_trace=eps_tr, x_trace=x_tr, use_graph=False)
    ref = x_T.clone()
    for k, (t, on_late) in enumerate(zip(ts, fl)):
        e = _guided_eps(late if on_late else early, ref, t, y, null, s)
        assert torch.equal(eps_tr[k], e), (pair, rule, t)
        lib.check(L.ddb_ddpm_step(ref.data_ptr(), e.data_ptr(), noise[t].data_ptr(), coef.data_ptr(), t, mode, 0,
                                  ref.numel(), lib.current_stream_ptr()))
        assert torch.equal(x_tr[k], ref), (pair, rule, t)
    assert torch.equal(x, ref)


# ------------------------------------------------------------------------------------------------ graph / s = 0
def test_graph_replay_equals_eager_steps(dev):
    """A whole DDPM trajectory (DuoDiff, Philox noise) and a DDIM trajectory: captured graphs == eager, bit for bit."""
    from duodiff_b200.ddpm import Sampler
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model("imagenet64_3", 43, True, dev), _model("imagenet64", 44, True, dev)
    B = 2
    g = torch.Generator(device=dev).manual_seed(6)
    x_T = torch.randn(B, 3, 64, 64, device=dev, generator=g)
    y = torch.tensor([5, 17], device=dev)
    smp = Sampler(early.engine(2 * B), late.engine(2 * B), 300, B, guidance=(SCALE, _null(early)))
    a, b = x_T.clone(), x_T.clone()
    smp.run(a, y=y, seed=9, use_graph=True)
    smp.run(b, y=y, seed=9, use_graph=False)
    assert torch.equal(a, b) and bool(torch.isfinite(a).all())
    steps, flags = _ddim_plan(50, True, 300)
    smp = Sampler(early.engine(2 * B), late.engine(2 * B), 300, B, rule=("ddim", 50, 0.0), guidance=(SCALE, 999))
    a, b = x_T.clone(), x_T.clone()
    smp.run_list(a, steps, flags, y=y, seed=9, use_graph=True)
    smp.run_list(b, steps, flags, y=y, seed=9, use_graph=False)
    assert torch.equal(a, b)


@pytest.mark.parametrize("use_ddim", [False, True])
def test_scale_zero_is_unguided_bit_for_bit(dev, use_ddim):
    """cfg_scale = 0: c + 0 * (c - u) == c, and the conditional half of the 2B-row forward is the B-row forward
    (batch invariance): samples and timesteps_save intermediates equal the unguided run."""
    from duodiff_b200 import sampler as S
    early, late = _model("imagenet256_3", 45, True, dev), _model("imagenet256", 46, True, dev)
    y = torch.tensor([1, 500, 999])
    kw = dict(batch_size=3, postprocessing=S.predict_noise_postprocessing, seed=2, num_channels=4, sample_height=32,
              sample_width=32, use_ddim=use_ddim, ddim_steps=20, ddim_eta=0.05, y=y, late_model=late, t_switch=300,
              timesteps_save=[1, 900] if use_ddim else [1, 500, 900])
    out0, inter0 = S.get_samples(early, **kw)
    out1, inter1 = S.get_samples(early, cfg_scale=0.0, **kw)
    assert np.array_equal(out0, out1)
    assert len(inter0) == len(inter1) > 0
    for a, b in zip(inter0, inter1):
        assert np.array_equal(a, b)
    out2, _ = S.get_samples(early, cfg_scale=SCALE, **kw)  # and a nonzero scale changes the samples
    assert float(np.abs(out2 - out0).max()) > 1e-3


# ------------------------------------------------------------------------------------------------ oracle
def test_free_running_guided_trajectory_matches_the_oracle(dev):
    from duodiff_b200.ddpm import Sampler
    net = _model("imagenet256_3", 47, False, dev)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    spec = O.UViTSpec.from_params(CONFIGS["imagenet256_3"])
    B = 2
    g = torch.Generator().manual_seed(7)
    x_T = torch.randn(B, 4, 32, 32, generator=g).to(dev)
    noise = torch.randn(1000, B, 4, 32, 32, generator=g).to(dev)
    y = torch.tensor([3, 640], device=dev)
    f = lambda x, t, yy: O.uvit_forward(sd, spec, x, t, yy)  # noqa: E731
    ref = G.sample_ddpm_guided(f, None, np.inf, x_T.clone(), noise, y, SCALE, 1000)
    x = x_T.clone()
    Sampler(net.engine(2 * B), None, np.inf, B, guidance=(SCALE, 1000)).run(x, y=y, noise=noise)
    r = rel_l2(x, ref)
    unguided = O.sample_ddpm(f, None, np.inf, x_T.clone(), noise, y=y)
    print(f"guided free-running final x rel-L2 {r:.2e} (bound {IMG_REL_L2_GUIDED:.1e}); "
          f"guided vs unguided oracle {rel_l2(ref, unguided):.2e}")
    assert r <= IMG_REL_L2_GUIDED
    assert not torch.equal(ref, unguided)


# ------------------------------------------------------------------------------------------------ batch / shards
def test_batch_invariance_and_shards(dev):
    from duodiff_b200 import sampler as S
    from duodiff_b200.ddpm import Sampler
    net = _model("imagenet64_3", 48, True, dev)
    B = 4
    g = torch.Generator(device=dev).manual_seed(8)
    x_T = torch.randn(B, 3, 64, 64, device=dev, generator=g)
    noise = torch.randn(1000, B, 3, 64, 64, device=dev, generator=g)
    y = torch.tensor([7, 70, 700, 998], device=dev)
    whole = x_T.clone()
    Sampler(net.engine(2 * B), None, np.inf, B, guidance=(SCALE, 999)).run(whole, y=y, noise=noise, t_first=999,
                                                                           t_last=950)
    for b in (0, 2):  # sample b alone, injected noise
        one = x_T[b:b + 1].clone()
        Sampler(net.engine(2 * B), None, np.inf, 1, guidance=(SCALE, 999)).run(
            one, y=y[b:b + 1], noise=noise[:, b:b + 1].contiguous(), t_first=999, t_last=950)
        assert torch.equal(one, whole[b:b + 1]), b
    # Philox noise keyed by the global row: shards with noise_row_offset == the whole guided batch
    kw = dict(postprocessing=S.predict_noise_postprocessing, seed=4, num_channels=3, sample_height=64, sample_width=64,
              use_ddim=True, ddim_steps=20, cfg_scale=SCALE)
    torch.manual_seed(4)
    x_all = torch.randn(B, 3, 64, 64)
    full, _ = S.get_samples(net, B, y=y.cpu(), x_T=x_all, **kw)
    for lo, hi in ((0, 1), (1, 4)):
        part, _ = S.get_samples(net, hi - lo, y=y[lo:hi].cpu(), x_T=x_all[lo:hi], noise_row_offset=lo, **kw)
        assert np.array_equal(part, full[lo:hi]), (lo, hi)


# ------------------------------------------------------------------------------------------------ rejections
def test_c_level_rejections(dev):
    import duodiff_b200 as ddb
    from duodiff_b200 import sampler as S
    from duodiff_b200._lib import DuoDiffError
    from duodiff_b200.ddpm import Sampler
    cond = _model("imagenet64_3", 49, False, dev)
    with pytest.raises(DuoDiffError, match="max_batch"):
        Sampler(ddb.UViT(**CONFIGS["imagenet64_3"]).to(dev).engine(3), None, np.inf, 2, guidance=(1.0, 999))
    with pytest.raises(DuoDiffError, match="class-conditional"):
        Sampler(_model("cifar10_3", 50, False, dev).engine(4), None, np.inf, 2, guidance=(1.0, 0))
    with pytest.raises(DuoDiffError, match="outside"):
        Sampler(cond.engine(4), None, np.inf, 2, guidance=(1.0, 1000))
    with pytest.raises(DuoDiffError, match="not finite"):
        Sampler(cond.engine(4), None, np.inf, 2, guidance=(float("nan"), 999))
    torch.manual_seed(0)
    ee = ddb.EarlyExitUViT(ddb.UViT(**CONFIGS["imagenet64_3"]), "mlp_probe_per_layer").eval().to(dev)
    with pytest.raises(DuoDiffError, match="early exit"):
        Sampler(ee.engine(4), None, np.inf, 2, ee_threshold=0.3, ee_mode=1, guidance=(1.0, 999))
    with pytest.raises(ValueError, match="early exit"):
        S.get_samples(ee, 2, S.predict_noise_postprocessing, 0, 3, 64, 64, y=torch.tensor([1, 2]), cfg_scale=1.0)
    with pytest.raises(ValueError, match="needs class labels"):
        S.get_samples(cond, 2, S.predict_noise_postprocessing, 0, 3, 64, 64, cfg_scale=1.0)


# ------------------------------------------------------------------------------------------------ command line
def _first_gpu_only():
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    return dict(os.environ, CUDA_VISIBLE_DEVICES=visible.split(",")[0] if visible else "0")


def _run(cmd, env=None, timeout=900):
    rc, out = run_tree(cmd, timeout, cwd=ROOT, env=env)
    if rc is None:
        pytest.fail(f"timed out after {timeout} s: {' '.join(cmd)}\n{out[-4000:]}")
    if rc != 0:
        pytest.fail(f"exit code {rc}: {' '.join(cmd)}\n{out[-4000:]}")
    return out


def _cli_args(tmp):
    from tests.test_gpu_cli import _write
    ck, cfg = _write(tmp, "in64", CONFIGS["imagenet64_3"], 5, wrap=True)
    return ["--checkpoint_path", ck, "--config_path", cfg, "--batch_size", "3", "--parametrization", "predict_noise",
            "--use_ddim", "--ddim_steps", "20", "--class_id", "1", "--cfg_scale", "0.4", "--seed", "1"]


def test_cli_writes_guided_samples(tmp_path, capsys):
    from duodiff_b200 import sampler as S
    out = tmp_path / "out"
    S.main(_cli_args(tmp_path) + ["--output_folder", str(out)])
    assert "null label 999" in capsys.readouterr().out
    names = sorted(p.name for p in out.iterdir())
    assert names == ["0.png", "1.png", "2.png", "grid_image.png", "statistics.txt"]
    assert (out / "statistics.txt").read_text().startswith("Elapsed time: ")


def test_cli_guided_under_torchrun_is_byte_identical(tmp_path):
    args = _cli_args(tmp_path)
    single, multi = tmp_path / "single", tmp_path / "torchrun2"
    env = _first_gpu_only()
    _run([sys.executable, "sampler.py", *args, "--output_folder", str(single)], env=env)
    out = _run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2", "sampler.py",
                *args, "--output_folder", str(multi)], env=env)
    assert "Gathered" in out and "null label 999" in out
    names = sorted(p.name for p in single.iterdir())
    assert names == sorted(p.name for p in multi.iterdir()) and "0.png" in names
    for name in names:
        if name != "statistics.txt":
            assert (single / name).read_bytes() == (multi / name).read_bytes(), name
