"""GPU tests of UniPC (`-m gpu`, B200): the predictor-corrector step tail (step_tail_kernel<C, W, G, TAIL_UNIPC>), the
sampler's history buffers (corrected x, D1, D2), `get_samples(unipc_steps=...)` and `sampler.py --unipc_steps`.

The tail rounds every operation on its own, so each step is checked bit for bit against torch:
    D = a*x + b*eps;  xc = x | ((cx*xb + c0*D) + c1*D1) [+ c2*D2];  x' = (px*xc + p0*D) [+ p1*D1];
    xb <- xc, D2 <- D1, D1 <- D.

Oracle parity (test_free_running_trajectory_matches_the_oracle): reference-init ImageNet-256 depth-3 backbone, the
20-point grid (19 evaluations), fp32 structured oracle (oracle/unipc_oracle.py, TF32 off).  x' depends on the data
predictions of the last three steps with the weights px*c0 + p0, px*c1 + p1 and px*c2; a DDIM step has the single
weight p0 + p1 (= -alpha_s expm1(-h)).  So a step's x' error is the eps error times the ratio w of the summed absolute
weights to that one, and the unguided bound for reference-init weights (5e-3, test_gpu_parity.py) becomes 5e-3 *
max w = 5e-3 * 2.56 = 1.3e-2 on this grid; guided (s = 0.4) that times (1 + 2s) (test_gpu_guidance.py).  Measured on
a B200: see the printed values (recorded in DESIGN.md section 3c).
"""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import guidance_oracle as G
from oracle import unipc_oracle as U
from oracle import uvit_oracle as O
from tests.helpers import CONFIGS, heat_, rel_l2
from tests.process_tree import run_tree

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
SCALE = 0.4


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


def _eps(net, x, t, y, s):
    """The model output the tail uses: one forward, or the guided composition c + s (c - u) on 2B rows."""
    B = x.shape[0]
    if s is None:
        return net(x, torch.full((B,), float(t), device=x.device), y)
    null = net.num_classes - 1
    out = net(torch.cat([x, x]), torch.full((2 * B,), float(t), device=x.device),
              torch.cat([y, torch.full_like(y, null)]))
    c, u = out[:B], out[B:]
    return c + s * (c - u)


def _torch_step(row, x, e, xb, d1, d2):
    """The kernel's update as separately rounded torch ops; returns (x', xc, D, the new D2)."""
    a, b, cx, c0, c1, c2, px, p0, p1 = (row[i] for i in range(9))
    corr, pred = int(row[9]), int(row[10])
    d = (a * x) + (b * e)
    xc = x
    if corr >= 1:
        xc = ((cx * xb) + (c0 * d)) + (c1 * d1)
        if corr == 2:
            xc = xc + (c2 * d2)
    o = (px * xc) + (p0 * d)
    if pred == 2:
        o = o + (p1 * d1)
    return o, xc, d, d1 if corr >= 1 else d2


def _weights(table):
    """Per grid row: summed absolute weights of D_k, D_{k-1}, D_{k-2} in x' over the DDIM step's weight."""
    t = table.double()
    rows = t[t[:, 10] > 0]
    px, c0, c1, c2, p0, p1 = rows[:, 6], rows[:, 3], rows[:, 4], rows[:, 5], rows[:, 7], rows[:, 8]
    return ((px * c0 + p0).abs() + (px * c1 + p1).abs() + (px * c2).abs()) / (p0 + p1).abs()


def _sampler(early, late, B, n, rule="predict_noise", s=None):
    from duodiff_b200.ddpm import Sampler
    rows = B if s is None else 2 * B
    guidance = None if s is None else (s, early.num_classes - 1)
    return Sampler(early.engine(rows), late.engine(rows) if late is not None else None, 300, B,
                   rule=("unipc", n, rule), guidance=guidance)


# ------------------------------------------------------------------------------------------------ composition
@pytest.mark.parametrize("pair", [("imagenet64_3", "imagenet64"), ("imagenet256_3", "imagenet256")])
@pytest.mark.parametrize("rule", ["predict_noise", "predict_original"])
@pytest.mark.parametrize("s", [None, 1.75])
def test_step_is_the_torch_composition_bit_for_bit(dev, pair, rule, s):
    """The whole 10-point grid (9 evaluations, eager, traced): corrector orders 0, 1 and 2, predictor orders 1 and 2,
    the hand-off after t = 666.  The sampler's history is first filled with NaN by a run from a NaN x_T: the first
    row (corrector 0) and the second (corrector 1, no D2) must not read what they do not use."""
    from duodiff_b200.ddpm import unipc_coefficients
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model(pair[0], 51, True, dev), _model(pair[1], 52, True, dev)
    B, C, H = 3, early.in_chans, early.img_size
    g = torch.Generator(device=dev).manual_seed(5)
    x_T = torch.randn(B, C, H, H, device=dev, generator=g)
    y = torch.randint(0, early.num_classes - 1, (B,), device=dev, generator=g)
    n = 10
    ts, fl = _ddim_plan(n, True, 300)
    assert any(fl) and not all(fl)
    table = unipc_coefficients(n, rule)[0].to(dev)
    assert [int(table[t, 9]) for t in ts] == [0, 1] + [2] * 7 and [int(table[t, 10]) for t in ts] == [1] + [2] * 7 + [1]
    smp = _sampler(early, late, B, n, rule, s)
    poison = torch.full_like(x_T, float("nan"))
    smp.run_list(poison, ts, fl, y=y, use_graph=False)
    assert bool(torch.isnan(poison).all())
    eps_tr, x_tr = torch.zeros(len(ts), B, C, H, H, device=dev), torch.zeros(len(ts), B, C, H, H, device=dev)
    x = x_T.clone()
    smp.run_list(x, ts, fl, y=y, eps_trace=eps_tr, x_trace=x_tr, use_graph=False)
    ref = x_T.clone()
    xb, d1, d2 = (torch.full_like(x_T, float("nan")) for _ in range(3))
    for k, (t, on_late) in enumerate(zip(ts, fl)):
        e = _eps(late if on_late else early, ref, t, y, s)
        assert torch.equal(eps_tr[k], e), (pair, rule, s, t)
        ref, xb, d, d2 = _torch_step(table[t], ref, eps_tr[k], xb, d1, d2)
        d1 = d
        assert torch.equal(x_tr[k], ref), (pair, rule, s, t)
    assert torch.equal(x, ref) and bool(torch.isfinite(x).all())


# ------------------------------------------------------------------------------------------------ graph / segments
def test_graph_replay_equals_eager(dev):
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model("imagenet64_3", 53, True, dev), _model("imagenet64", 54, True, dev)
    B = 2
    x_T = torch.randn(B, 3, 64, 64, device=dev, generator=torch.Generator(device=dev).manual_seed(6))
    y = torch.tensor([5, 17], device=dev)
    steps, flags = _ddim_plan(20, True, 300)
    for s in (None, SCALE):
        smp = _sampler(early, late, B, 20, s=s)
        a, b = x_T.clone(), x_T.clone()
        smp.run_list(a, steps, flags, y=y, use_graph=True)
        smp.run_list(b, steps, flags, y=y, use_graph=False)
        assert torch.equal(a, b) and bool(torch.isfinite(a).all()), s


def test_timesteps_save_segments_equal_one_run(dev):
    """get_samples cuts the trajectory at the saved steps; the history carries across the segments."""
    from duodiff_b200 import sampler as S
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model("imagenet256_3", 55, True, dev), _model("imagenet256", 56, True, dev)
    y = torch.tensor([1, 500, 999])
    kw = dict(batch_size=3, postprocessing=S.predict_noise_postprocessing, seed=2, num_channels=4, sample_height=32,
              sample_width=32, y=y, late_model=late, t_switch=300, unipc_steps=20)
    out0, inter0 = S.get_samples(early, **kw)
    save = [1000 - 946, 1000 - 473, 1000 - 52]  # after the steps at t = 946, 473 and 52 (grid points)
    out1, inter1 = S.get_samples(early, timesteps_save=save, **kw)
    assert np.array_equal(out0, out1) and len(inter1) == 3
    steps, flags = _ddim_plan(20, True, 300)
    torch.manual_seed(2)
    x = torch.randn(3, 4, 32, 32).to(dev)
    x_tr = torch.zeros(len(steps), 3, 4, 32, 32, device=dev)
    smp = _sampler(early, late, 3, 20)
    smp.run_list(x, steps, flags, y=y.to(dev), x_trace=x_tr, use_graph=False)
    for got, t in zip(inter1, (946, 473, 52)):
        want = smp.finalize(x_tr[steps.index(t)].contiguous()).cpu().numpy()
        assert np.array_equal(got, want), t
    assert np.array_equal(out0, smp.finalize(x).cpu().numpy())


def test_cached_sampler_restarts_the_history(dev):
    from duodiff_b200 import sampler as S
    net = _model("imagenet64_3", 57, True, dev)
    kw = dict(batch_size=2, postprocessing=S.predict_original_postprocessing, num_channels=3, sample_height=64,
              sample_width=64, y=torch.tensor([3, 4]), unipc_steps=12)
    a, _ = S.get_samples(net, seed=1, **kw)
    b, _ = S.get_samples(net, seed=2, **kw)
    c, _ = S.get_samples(net, seed=1, **kw)
    assert np.array_equal(a, c) and not np.array_equal(a, b)


# ------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("s", [None, SCALE])
def test_free_running_trajectory_matches_the_oracle(dev, s):
    from duodiff_b200.ddpm import unipc_coefficients
    from duodiff_b200.sampler import _ddim_plan
    net = _model("imagenet256_3", 58, False, dev)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    spec = O.UViTSpec.from_params(CONFIGS["imagenet256_3"])
    B, n = 2, 20
    g = torch.Generator().manual_seed(7)
    x_T = torch.randn(B, 4, 32, 32, generator=g).to(dev)
    y = torch.tensor([3, 640], device=dev)
    f = lambda x, t, yy: O.uvit_forward(sd, spec, x, t, yy)  # noqa: E731
    if s is not None:
        f = G.guided_model(f, s, 1000)
    ref = U.sample_unipc(f, None, np.inf, x_T.clone(), n, y=y)
    x = x_T.clone()
    steps, flags = _ddim_plan(n, False, np.inf)
    _sampler(net, None, B, n, s=s).run_list(x, steps, flags, y=y)
    w = float(_weights(unipc_coefficients(n)[0]).max())
    bound = 5e-3 * w * (1 if s is None else 1 + 2 * s)
    r = rel_l2(x, ref)
    print(f"UniPC 20-point free-running x_0 rel-L2 {r:.2e} (bound {bound:.1e}, max weight ratio {w:.2f}), "
          f"guidance {s}")
    assert r <= bound


# ------------------------------------------------------------------------------------------------ batch / shards
def test_batch_invariance(dev):
    from duodiff_b200.sampler import _ddim_plan
    net = _model("imagenet64_3", 59, True, dev)
    B = 4
    x_T = torch.randn(B, 3, 64, 64, device=dev, generator=torch.Generator(device=dev).manual_seed(8))
    y = torch.tensor([7, 70, 700, 998], device=dev)
    steps, flags = _ddim_plan(15, False, np.inf)
    whole = x_T.clone()
    _sampler(net, None, B, 15, s=SCALE).run_list(whole, steps, flags, y=y)
    for b in (0, 2):
        one = x_T[b:b + 1].clone()
        _sampler(net, None, 1, 15, s=SCALE).run_list(one, steps, flags, y=y[b:b + 1])
        assert torch.equal(one, whole[b:b + 1]), b


def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def _shard_worker(rank, world, port, flag):
    import torch.distributed as dist

    from duodiff_b200 import distributed as D
    from duodiff_b200 import sampler as S
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        dev = torch.device("cuda:0")
        torch.cuda.set_device(dev)
        net = _model("imagenet64_3", 60, True, dev)
        y = torch.tensor([1, 2, 3, 4, 5])
        kw = dict(postprocessing=S.predict_noise_postprocessing, num_channels=3, sample_height=64, sample_width=64,
                  unipc_steps=20, cfg_scale=SCALE)
        got = D.get_samples_sharded(lambda **k: S.get_samples(net, **k, **kw), 5, shape=(3, 64, 64), y=y, seed=3)
        if rank == 0:
            whole, _ = S.get_samples(net, 5, seed=3, y=y, **kw)
            assert np.array_equal(got.cpu().numpy(), whole)
            open(flag, "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_two_shards_on_one_gpu_equal_the_whole_batch(tmp_path):
    import torch.multiprocessing as mp
    flag = tmp_path / "ok"
    mp.spawn(_shard_worker, args=(2, _free_port(), str(flag)), nprocs=2, join=True)
    assert flag.read_text() == "ok"


# ------------------------------------------------------------------------------------------------ rejections
def test_c_level_rejections(dev):
    import duodiff_b200 as ddb
    from duodiff_b200 import _lib
    from duodiff_b200._lib import DuoDiffError
    from duodiff_b200.ddpm import Sampler, unipc_coefficients
    torch.manual_seed(0)
    ee = ddb.EarlyExitUViT(ddb.UViT(**CONFIGS["imagenet64_3"]), "mlp_probe_per_layer").eval().to(dev)
    with pytest.raises(DuoDiffError, match="early exit"):
        Sampler(ee.engine(2), None, np.inf, 2, rule=("unipc", 20, "predict_noise"), ee_threshold=0.3, ee_mode=1)
    L = _lib.load()
    x, e = torch.zeros(2, 3, 64, 64, device=dev), torch.zeros(2, 3, 64, 64, device=dev)
    coef = unipc_coefficients(20)[0].to(dev)
    with pytest.raises(DuoDiffError, match="mode 4"):
        _lib.check(L.ddb_ddpm_step(x.data_ptr(), e.data_ptr(), None, coef.data_ptr(), 999, 4, 0, x.numel(),
                                   _lib.current_stream_ptr()))
    net = _model("imagenet64_3", 61, False, dev)
    smp = _sampler(net, None, 2, 20)
    y = torch.tensor([1, 2], device=dev)
    with pytest.raises(DuoDiffError, match="not a step of the UniPC"):
        smp.run_list(x, [999, 998], [False, False], y=y)
    with pytest.raises(DuoDiffError, match="not a step of the UniPC"):
        smp.run_list(x, [0], [False], y=y)  # the grid's end point: no step starts there
    with pytest.raises(DuoDiffError, match="not a step of the UniPC"):
        smp.profile_step(x, 500, False, y=y)
    with pytest.raises(DuoDiffError, match="run_list"):
        smp.run(x, y=y)
    smp.profile_step(x, 999, False, y=y)  # a grid step profiles


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


def _cli_args(tmp, guided=True):
    from tests.test_gpu_cli import _write
    ck, cfg = _write(tmp, "in64", CONFIGS["imagenet64_3"], 5, wrap=True)
    return ["--checkpoint_path", ck, "--config_path", cfg, "--batch_size", "3", "--parametrization", "predict_noise",
            "--unipc_steps", "16", "--class_id", "1", "--seed", "1"] + (["--cfg_scale", "0.4"] if guided else [])


def test_cli_writes_unipc_samples(tmp_path):
    from duodiff_b200 import sampler as S
    out = tmp_path / "out"
    S.main(_cli_args(tmp_path) + ["--output_folder", str(out)])
    assert sorted(p.name for p in out.iterdir()) == ["0.png", "1.png", "2.png", "grid_image.png", "statistics.txt"]
    out = tmp_path / "saved"
    S.main(_cli_args(tmp_path, guided=False) + ["--timesteps_save", "68", "534", "--output_folder", str(out)])
    names = sorted(p.name for p in out.iterdir())
    assert "0.png" in names and len(names) > 5


def test_cli_under_torchrun_is_byte_identical(tmp_path):
    args = _cli_args(tmp_path) + ["--timesteps_save", "68"]
    single, multi = tmp_path / "single", tmp_path / "torchrun2"
    env = _first_gpu_only()
    _run([sys.executable, "sampler.py", *args, "--output_folder", str(single)], env=env)
    out = _run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2", "sampler.py",
                *args, "--output_folder", str(multi)], env=env)
    assert "Gathered" in out
    names = sorted(p.name for p in single.iterdir())
    assert names == sorted(p.name for p in multi.iterdir()) and "0.png" in names
    for name in names:
        if name != "statistics.txt":
            assert (single / name).read_bytes() == (multi / name).read_bytes(), name
