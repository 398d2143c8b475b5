"""GPU tests of SDE-DPM-Solver++(2M) (`-m gpu`, B200): the stochastic multistep step tail (step_tail_kernel<C, W, G,
TAIL_SDE2M>), the sampler's D_prev buffer, `get_samples(sde_dpm_solver_steps=...)` and
`sampler.py --sde_dpm_solver_steps`.

The tail rounds every operation on its own, so each step is checked bit for bit against torch:
    D_t = a*x + b*eps;  D = w0*D_t + w1*D_prev (order 2) | D_t;  x' = (rho*x + phi*D) [+ vs*z where vs != 0];
    D_prev <- D_t.
z is the DDPM tail's draw at t: the injected noise[t], or the Philox draw that ddb_ddpm_step makes at (seed, t).

Oracle parity (test_free_running_trajectory_matches_the_oracle): reference-init ImageNet-256 depth-3 backbone, the
20-point grid (19 evaluations), fp32 textbook oracle (oracle/sde_dpm_solver_oracle.py, TF32 off), the same injected
noise.  x' depends on the data predictions of the last two steps with the weights phi*w0 and phi*w1; a first-order
step has the single weight phi.  So a step's x' error is the eps error times w = |w0| + |w1|, and the unguided bound
for reference-init weights (5e-3, test_gpu_parity.py) becomes 5e-3 * max w on this grid; guided (s = 0.4) that times
(1 + 2s) (test_gpu_guidance.py).  The noise term adds no error: z is the same tensor on both sides.  Measured on a
B200: see the printed values (recorded in DESIGN.md section 3c).
"""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import guidance_oracle as G
from oracle import sde_dpm_solver_oracle as SO
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


def _torch_step(row, x, e, d_prev, z):
    """The kernel's update as separately rounded torch ops; returns (x', D_t)."""
    a, b, rho, phi, w0, w1 = (row[i] for i in range(6))
    dt = (a * x) + (b * e)
    d = ((w0 * dt) + (w1 * d_prev)) if int(row[6]) == 2 else dt
    o = (rho * x) + (phi * d)
    if float(row[7]) != 0:
        o = o + (row[7] * z)
    return o, dt


def _ddpm_draw(x_like, t, seed):
    """The Philox z of the DDPM step at t: ddb_ddpm_step in mode 1 with the row {0, 0, 1, 0} gives x' = (0*out + 0*x)
    + 1*z = z."""
    from duodiff_b200 import _lib
    L = _lib.load()
    coef = torch.zeros(1000, 4, device=x_like.device)
    coef[t, 2] = 1.0
    z, out = torch.zeros_like(x_like), torch.zeros_like(x_like)
    _lib.check(L.ddb_ddpm_step(z.data_ptr(), out.data_ptr(), None, coef.data_ptr(), int(t), 1, int(seed), z.numel(),
                               _lib.current_stream_ptr()))
    return z


def _weights(table):
    """Per grid row: |w0| + |w1|, the summed weight of the data predictions in x' over a first-order step's."""
    t = table.double()
    rows = t[t[:, 6] > 0]
    return rows[:, 4].abs() + rows[:, 5].abs()


def _sampler(early, late, B, n, rule="predict_noise", s=None):
    from duodiff_b200.ddpm import Sampler
    rows = B if s is None else 2 * B
    guidance = None if s is None else (s, early.num_classes - 1)
    return Sampler(early.engine(rows), late.engine(rows) if late is not None else None, 300, B,
                   rule=("sde-dpm_solver++", n, rule), guidance=guidance)


# ------------------------------------------------------------------------------------------------ composition
@pytest.mark.parametrize("pair", [("imagenet64_3", "imagenet64"), ("imagenet256_3", "imagenet256")])
@pytest.mark.parametrize("rule", ["predict_noise", "predict_original"])
@pytest.mark.parametrize("s", [None, 1.75])
def test_step_is_the_torch_composition_bit_for_bit(dev, pair, rule, s):
    """The whole 10-point grid (9 evaluations, eager, traced, injected noise): order 1, 2, ..., 2, 1, the hand-off
    after t = 666 and the noise-free final step.  D_prev is first filled with NaN by a run from a NaN x_T: the
    order-1 first row must not read it."""
    from duodiff_b200.ddpm import sde_dpm_solver_coefficients
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model(pair[0], 51, True, dev), _model(pair[1], 52, True, dev)
    B, C, H = 3, early.in_chans, early.img_size
    g = torch.Generator(device=dev).manual_seed(5)
    x_T = torch.randn(B, C, H, H, device=dev, generator=g)
    y = torch.randint(0, early.num_classes - 1, (B,), device=dev, generator=g)
    noise = torch.randn(1000, B, C, H, H, device=dev, generator=g)
    n = 10
    ts, fl = _ddim_plan(n, True, 300)
    assert any(fl) and not all(fl)
    table = sde_dpm_solver_coefficients(n, rule)[0].to(dev)
    assert [int(table[t, 6]) for t in ts] == [1] + [2] * 7 + [1]
    smp = _sampler(early, late, B, n, rule, s)
    poison = torch.full_like(x_T, float("nan"))
    smp.run_list(poison, ts, fl, y=y, noise=noise, use_graph=False)
    assert bool(torch.isnan(poison).all())
    eps_tr, x_tr = torch.zeros(len(ts), B, C, H, H, device=dev), torch.zeros(len(ts), B, C, H, H, device=dev)
    x = x_T.clone()
    smp.run_list(x, ts, fl, y=y, noise=noise, eps_trace=eps_tr, x_trace=x_tr, use_graph=False)
    ref, d_prev = x_T.clone(), torch.full_like(x_T, float("nan"))
    for k, (t, on_late) in enumerate(zip(ts, fl)):
        e = _eps(late if on_late else early, ref, t, y, s)
        assert torch.equal(eps_tr[k], e), (pair, rule, s, t)
        ref, d_prev = _torch_step(table[t], ref, eps_tr[k], d_prev, noise[t])
        assert torch.equal(x_tr[k], ref), (pair, rule, s, t)
    assert torch.equal(x, ref) and bool(torch.isfinite(x).all())


@pytest.mark.parametrize("s", [None, SCALE])
def test_philox_noise_is_the_ddpm_draw(dev, s):
    """Without injected noise each step adds vs * z with z the DDPM tail's Philox draw at the same (seed, t, element)."""
    from duodiff_b200.ddpm import sde_dpm_solver_coefficients
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model("imagenet64_3", 62, True, dev), _model("imagenet64", 63, True, dev)
    B, seed = 2, 12345
    x_T = torch.randn(B, 3, 64, 64, device=dev, generator=torch.Generator(device=dev).manual_seed(9))
    y = torch.tensor([11, 22], device=dev)
    ts, fl = _ddim_plan(12, True, 300)
    table = sde_dpm_solver_coefficients(12)[0].to(dev)
    eps_tr, x_tr = torch.zeros(len(ts), *x_T.shape, device=dev), torch.zeros(len(ts), *x_T.shape, device=dev)
    x = x_T.clone()
    _sampler(early, late, B, 12, s=s).run_list(x, ts, fl, y=y, seed=seed, eps_trace=eps_tr, x_trace=x_tr,
                                               use_graph=False)
    ref, d_prev = x_T.clone(), torch.full_like(x_T, float("nan"))
    for k, t in enumerate(ts):
        ref, d_prev = _torch_step(table[t], x_tr[k - 1] if k else x_T, eps_tr[k], d_prev, _ddpm_draw(x_T, t, seed))
        assert torch.equal(x_tr[k], ref), (s, t)
    assert torch.equal(x, x_tr[-1])


# ------------------------------------------------------------------------------------------------ graph / segments
def test_graph_replay_equals_eager(dev):
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model("imagenet64_3", 53, True, dev), _model("imagenet64", 54, True, dev)
    B = 2
    g = torch.Generator(device=dev).manual_seed(6)
    x_T = torch.randn(B, 3, 64, 64, device=dev, generator=g)
    noise = torch.randn(1000, B, 3, 64, 64, device=dev, generator=g)
    y = torch.tensor([5, 17], device=dev)
    steps, flags = _ddim_plan(20, True, 300)
    for s in (None, SCALE):
        smp = _sampler(early, late, B, 20, s=s)
        for z in (None, noise):
            a, b = x_T.clone(), x_T.clone()
            smp.run_list(a, steps, flags, y=y, noise=z, seed=4, use_graph=True)
            smp.run_list(b, steps, flags, y=y, noise=z, seed=4, use_graph=False)
            assert torch.equal(a, b) and bool(torch.isfinite(a).all()), (s, z is None)


def test_timesteps_save_segments_equal_one_run(dev):
    """get_samples cuts the trajectory at the saved steps; D_prev carries across the segments, and a saved x is x
    after that step, its noise included."""
    from duodiff_b200 import sampler as S
    from duodiff_b200.sampler import _ddim_plan
    early, late = _model("imagenet256_3", 55, True, dev), _model("imagenet256", 56, True, dev)
    y = torch.tensor([1, 500, 999])
    kw = dict(batch_size=3, postprocessing=S.predict_noise_postprocessing, seed=2, num_channels=4, sample_height=32,
              sample_width=32, y=y, late_model=late, t_switch=300, sde_dpm_solver_steps=20)
    out0, inter0 = S.get_samples(early, **kw)
    save = [1000 - 946, 1000 - 473, 1000 - 52]  # after the steps at t = 946, 473 and 52 (grid points)
    out1, inter1 = S.get_samples(early, timesteps_save=save, **kw)
    assert np.array_equal(out0, out1) and len(inter1) == 3
    steps, flags = _ddim_plan(20, True, 300)
    torch.manual_seed(2)
    x = torch.randn(3, 4, 32, 32).to(dev)
    x_tr = torch.zeros(len(steps), 3, 4, 32, 32, device=dev)
    smp = _sampler(early, late, 3, 20)
    smp.run_list(x, steps, flags, y=y.to(dev), seed=2, x_trace=x_tr, use_graph=False)
    for got, t in zip(inter1, (946, 473, 52)):
        want = smp.finalize(x_tr[steps.index(t)].contiguous()).cpu().numpy()
        assert np.array_equal(got, want), t
    assert np.array_equal(out0, smp.finalize(x).cpu().numpy())


def test_cached_sampler_restarts_the_history_and_seeds_select_the_noise(dev):
    """Same seed, same bits (the cached sampler's D_prev from another call does not leak); another seed draws other
    noise (and another x_T)."""
    from duodiff_b200 import sampler as S
    net = _model("imagenet64_3", 57, True, dev)
    kw = dict(batch_size=2, postprocessing=S.predict_original_postprocessing, num_channels=3, sample_height=64,
              sample_width=64, y=torch.tensor([3, 4]), sde_dpm_solver_steps=12)
    a, _ = S.get_samples(net, seed=1, **kw)
    b, _ = S.get_samples(net, seed=2, **kw)
    c, _ = S.get_samples(net, seed=1, **kw)
    assert np.array_equal(a, c) and not np.array_equal(a, b)
    # the same x_T with another Philox key: only the noise differs
    from duodiff_b200.sampler import _ddim_plan
    steps, flags = _ddim_plan(12, False, np.inf)
    smp = _sampler(net, None, 2, 12, rule="predict_original")
    x_T = torch.randn(2, 3, 64, 64, device=dev, generator=torch.Generator(device=dev).manual_seed(10))
    y = torch.tensor([3, 4], device=dev)
    u, v, w = x_T.clone(), x_T.clone(), x_T.clone()
    smp.run_list(u, steps, flags, y=y, seed=1)
    smp.run_list(v, steps, flags, y=y, seed=2)
    smp.run_list(w, steps, flags, y=y, seed=1)
    assert torch.equal(u, w) and not torch.equal(u, v)


# ------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("s", [None, SCALE])
def test_free_running_trajectory_matches_the_oracle(dev, s):
    from duodiff_b200.ddpm import sde_dpm_solver_coefficients
    from duodiff_b200.sampler import _ddim_plan
    net = _model("imagenet256_3", 58, False, dev)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    spec = O.UViTSpec.from_params(CONFIGS["imagenet256_3"])
    B, n = 2, 20
    g = torch.Generator().manual_seed(7)
    x_T = torch.randn(B, 4, 32, 32, generator=g).to(dev)
    noise = torch.randn(1000, B, 4, 32, 32, generator=g).to(dev)
    y = torch.tensor([3, 640], device=dev)
    f = lambda x, t, yy: O.uvit_forward(sd, spec, x, t, yy)  # noqa: E731
    if s is not None:
        f = G.guided_model(f, s, 1000)
    ref = SO.sample_sde_dpm_solver(f, None, np.inf, x_T.clone(), n, noise, y=y)
    x = x_T.clone()
    steps, flags = _ddim_plan(n, False, np.inf)
    _sampler(net, None, B, n, s=s).run_list(x, steps, flags, y=y, noise=noise)
    w = float(_weights(sde_dpm_solver_coefficients(n)[0]).max())
    bound = 5e-3 * w * (1 if s is None else 1 + 2 * s)
    r = rel_l2(x, ref)
    print(f"SDE-DPM-Solver++ 20-point free-running x_0 rel-L2 {r:.2e} (bound {bound:.1e}, max weight ratio {w:.2f}), "
          f"guidance {s}")
    assert r <= bound


# ------------------------------------------------------------------------------------------------ batch / shards
def test_batch_invariance(dev):
    """One sample run alone, with its noise offset, gives the bits it gets inside the batch (Philox noise)."""
    from duodiff_b200.sampler import _ddim_plan
    net = _model("imagenet64_3", 59, True, dev)
    B = 4
    x_T = torch.randn(B, 3, 64, 64, device=dev, generator=torch.Generator(device=dev).manual_seed(8))
    y = torch.tensor([7, 70, 700, 998], device=dev)
    steps, flags = _ddim_plan(15, False, np.inf)
    whole = x_T.clone()
    _sampler(net, None, B, 15, s=SCALE).run_list(whole, steps, flags, y=y, seed=6)
    for b in (0, 2):
        one = x_T[b:b + 1].clone()
        smp = _sampler(net, None, 1, 15, s=SCALE)
        smp.set_noise_offset(b)
        smp.run_list(one, steps, flags, y=y[b:b + 1], seed=6)
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
                  sde_dpm_solver_steps=20, cfg_scale=SCALE)
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
    from duodiff_b200.ddpm import Sampler, sde_dpm_solver_coefficients
    torch.manual_seed(0)
    ee = ddb.EarlyExitUViT(ddb.UViT(**CONFIGS["imagenet64_3"]), "mlp_probe_per_layer").eval().to(dev)
    with pytest.raises(DuoDiffError, match="early exit"):
        Sampler(ee.engine(2), None, np.inf, 2, rule=("sde-dpm_solver++", 20, "predict_noise"), ee_threshold=0.3,
                ee_mode=1)
    L = _lib.load()
    x, e = torch.zeros(2, 3, 64, 64, device=dev), torch.zeros(2, 3, 64, 64, device=dev)
    coef = sde_dpm_solver_coefficients(20)[0].to(dev)
    with pytest.raises(DuoDiffError, match="mode 5"):
        _lib.check(L.ddb_ddpm_step(x.data_ptr(), e.data_ptr(), None, coef.data_ptr(), 999, 5, 0, x.numel(),
                                   _lib.current_stream_ptr()))
    net = _model("imagenet64_3", 61, False, dev)
    smp = _sampler(net, None, 2, 20)
    y = torch.tensor([1, 2], device=dev)
    with pytest.raises(DuoDiffError, match="not a step of the SDE-DPM-Solver"):
        smp.run_list(x, [999, 998], [False, False], y=y)
    with pytest.raises(DuoDiffError, match="not a step of the SDE-DPM-Solver"):
        smp.run_list(x, [0], [False], y=y)  # the grid's end point: no step starts there
    with pytest.raises(DuoDiffError, match="not a step of the SDE-DPM-Solver"):
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
            "--sde_dpm_solver_steps", "16", "--class_id", "1", "--seed", "1"] + (["--cfg_scale", "0.4"] if guided else [])


def test_cli_writes_sde_dpm_solver_samples(tmp_path):
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
