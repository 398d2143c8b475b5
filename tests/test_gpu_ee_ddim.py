"""GPU tests of DDIM sampling with early exit (eesampler.get_samples(use_ddim=True), `eesampler.py --use_ddim`):
the two early-exit step paths on the strided grid, the composition of the steps, the logs against the oracle
(oracle/ee_ddim_oracle.py), the public API, sharding and the command line.

Note on eta: the reference's DDIM update (sampler.py:110-120) takes sqrt(1 - abar_s - eta * beta_tilde_t).  On the
last step (s = 0, 1 - abar_0 = 1e-4) that is negative for eta = 1 on the 20- and 50-point grids, so x_0 is NaN in the
reference as here.  The eta = 1 cases compare NaN-aware and also check the trajectory before that step."""
import functools
import os
import socket
import sys
from datetime import timedelta
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import uvit_oracle as O
from oracle.ee_ddim_oracle import ee_sample_ddim
from tests.helpers import CONFIGS, heat_, rel_l2

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]

EPS_REL_L2 = 2e-2
IMG_REL_L2 = 5e-3          # free-running, reference-init weights (tests/test_gpu_parity.py)
PROBE_MARGIN_HOT = 1.5e-2  # heat_()-ed probes (tests/test_gpu_parity.py)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda:0")


def _lib():
    from duodiff_b200 import _lib
    return _lib, _lib.load()


def _spread_probes(net, depth):
    """Random-init probes all sit near 0.5: spread them so that every exit layer occurs (as tests/test_gpu_parity.py)."""
    with torch.no_grad():
        for i in range(depth):
            net.matrix[f"{i}"].classifier[0].bias.fill_(1.5 - 3.0 * i / depth)


def _ee_net(name, seed, dev, ctype="mlp_probe_per_layer", hot=4.0, spread=True):
    """hot: heat_()'s Linear scale (0: reference init)."""
    import duodiff_b200 as ddb
    torch.manual_seed(seed)
    cfg = CONFIGS[name]
    net = ddb.EarlyExitUViT(ddb.UViT(**cfg), ctype)
    if hot:
        heat_(net, seed + 1, scale=hot)
    if spread:
        _spread_probes(net, cfg["depth"])
    return net.eval().to(dev)


def _grid(steps):
    from duodiff_b200.ddpm import ddim_timesteps
    return ddim_timesteps(steps)[:-1]


def _off_grid(steps):
    off = torch.ones(1000, dtype=torch.bool)
    off[_grid(steps)] = False
    return off


def _same(a, b):
    """Bit for bit, with NaN equal to NaN (tensors or numpy arrays)."""
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    return torch.equal(a.isnan(), b.isnan()) and torch.equal(torch.where(a.isnan(), 0, a), torch.where(b.isnan(), 0, b))


def _three_paths(fn):
    """fn(mode) under simulate (mode 0), the fused compaction step (mode 1) and the unfused compaction kernels
    (mode 1 with ee_fuse = 0)."""
    lib, L = _lib()
    r0, r1 = fn(0), fn(1)
    lib.check(L.ddb_set_option(b"ee_fuse", 0))
    try:
        r2 = fn(1)
    finally:
        lib.check(L.ddb_set_option(b"ee_fuse", 1))
    return r0, r1, r2


# ------------------------------------------------------------------------------------------------ 1. the three paths
@pytest.mark.parametrize("name", ["cifar10", "imagenet256_3"])
def test_compact_equals_simulate_on_the_grid(dev, name):
    from duodiff_b200 import eesampler as ES
    from duodiff_b200.ddpm import Sampler
    from duodiff_b200.sampler import _ddim_plan
    cfg = CONFIGS[name]
    depth, C, H = cfg["depth"], cfg["in_chans"], cfg["img_size"]
    net = _ee_net(name, 8, dev)
    B, thr = 5, 0.4
    g = torch.Generator().manual_seed(6)
    noise = torch.randn(1000, B, C, H, H, generator=g)
    y = torch.randint(0, cfg["num_classes"], (B,), generator=g).to(dev) if cfg["num_classes"] > 0 else None
    x_T = torch.randn(B, C, H, H, generator=g).to(dev)
    for steps in (20, 50):
        grid = _grid(steps)
        for eta in (0.0, 1.0):
            for injected in (True, False):
                kw = dict(seed=1, num_channels=C, sample_height=H, sample_width=H, threshold=thr, depth=depth, y=y,
                          noise=noise if injected else None, use_ddim=True, ddim_steps=steps, ddim_eta=eta)
                (s0, e0, i0), (s1, e1, i1), (s2, e2, i2) = _three_paths(lambda m: ES.get_samples(net, B, mode=m, **kw))
                case = (steps, eta, injected)
                assert _same(s0, s1) and _same(s1, s2), case
                assert torch.equal(i0[grid], i1[grid]) and torch.equal(i1[grid], i2[grid]), case
                assert _same(i0, i1) and _same(i1, i2) and _same(e1, e2), case
                assert float(i1[grid].min()) < depth, f"no early exits on the grid {case}"
                assert np.isfinite(s0).all() == (eta == 0.0), case  # eta = 1: the reference's last step is NaN
                if eta == 0.0:
                    continue
                # eta = 1: the trajectory up to the last step, where x is finite
                steps_, flags = _ddim_plan(steps, False, np.inf)

                def run(mode):
                    smp = Sampler(net.engine(B), None, np.inf, B, rule=("ddim", steps, eta), ee_threshold=thr,
                                  ee_mode=mode)
                    x = x_T.clone()
                    smp.run_list(x, steps_[:-1], flags[:-1], y=y, noise=noise.to(dev) if injected else None, seed=1)
                    return x
                x0, x1, x2 = _three_paths(run)
                assert torch.isfinite(x0).all() and torch.equal(x0, x1) and torch.equal(x1, x2), case


# ------------------------------------------------------------------------------------------------ 2. step composition
@pytest.mark.parametrize("mode", [0, 1])
def test_steps_compose_from_the_mode_2_update(dev, mode):
    """Eager run with eps / x traces through ddb_sampler_run_list_logs: each step's x is ddb_ddpm_step (mode 2) applied
    to the previous x and that step's selected eps, bit for bit; graph replay gives the eager bits and logs."""
    lib, L = _lib()
    from duodiff_b200.ddpm import Sampler, ddim_coefficients
    from duodiff_b200.sampler import _ddim_plan
    name = "celeba_3"
    cfg = CONFIGS[name]
    depth, C, H = cfg["depth"], cfg["in_chans"], cfg["img_size"]
    net = _ee_net(name, 40, dev)
    B, thr, steps = 4, 0.4, 20
    g = torch.Generator(device=dev).manual_seed(41)
    x_T = torch.randn(B, C, H, H, device=dev, generator=g)
    noise = torch.randn(1000, B, C, H, H, device=dev, generator=g)
    ts, flags = _ddim_plan(steps, False, np.inf)
    n = len(ts)
    for eta in (0.0, 1.0):
        table, m2 = ddim_coefficients(steps, eta)
        assert m2 == 2
        coef = table.to(dev)
        smp = Sampler(net.engine(B), None, np.inf, B, rule=("ddim", steps, eta), ee_threshold=thr, ee_mode=mode)
        for injected in (True, False):
            z = noise if injected else None
            x = x_T.clone()
            eps_tr, x_tr = torch.zeros(n, B, C, H, H, device=dev), torch.zeros(n, B, C, H, H, device=dev)
            ex = torch.full((1000, B), -7, dtype=torch.int32, device=dev)
            sc = torch.full((1000, depth), -7.0, device=dev)
            smp.run_list(x, ts, flags, noise=z, seed=9, eps_trace=eps_tr, x_trace=x_tr, exit_log=ex, score_log=sc,
                         use_graph=False)
            prev = x_T.clone()
            for k, t in enumerate(ts):
                ref = prev.clone()
                lib.check(L.ddb_ddpm_step(ref.data_ptr(), eps_tr[k].data_ptr(), noise[t].data_ptr() if injected else None,
                                          coef.data_ptr(), t, 2, 9, ref.numel(), lib.current_stream_ptr()))
                assert _same(ref, x_tr[k]), (eta, injected, t)
                prev = x_tr[k]
            assert _same(x, x_tr[-1])
            assert ex[ts].lt(depth).any(), "no early exits: the selected eps would all be the final head's"
            xg = x_T.clone()
            exg = torch.full((1000, B), -7, dtype=torch.int32, device=dev)
            scg = torch.full((1000, depth), -7.0, device=dev)
            smp.run_list(xg, ts, flags, noise=z, seed=9, exit_log=exg, score_log=scg, use_graph=True)
            assert _same(xg, x) and torch.equal(exg, ex) and _same(scg, sc), (eta, injected)
            off = _off_grid(steps).to(dev)
            assert exg[off].eq(-7).all() and scg[off].eq(-7.0).all()


# ------------------------------------------------------------------------------------------------ 3. logs vs oracle
def test_logs_teacher_forced_on_the_grid(dev):
    """Every grid step replayed on the oracle's own x_t: every index mismatch lies within the probe margin of the
    threshold, the batch-mean score rows match within the margin, and rows off the step keep the caller's sentinel."""
    from duodiff_b200.ddpm import Sampler
    net = _ee_net("cifar10", 8, dev)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    spec = O.UViTSpec.from_params(CONFIGS["cifar10"])
    B, thr, steps, eta = 4, 0.4, 20, 0.05
    g = torch.Generator().manual_seed(6)
    nz = torch.randn(1000, B, 3, 32, 32, generator=g).to(dev)
    x_T = torch.randn(B, 3, 32, 32, generator=g).to(dev)
    trace = {}
    model = lambda x, t, y: O.ee_forward(sd, spec, x, t, y)  # noqa: E731
    _x0, r_err, r_idx = ee_sample_ddim(model, thr, 13, x_T, nz, steps, eta, trace=trace)
    smp = Sampler(net.engine(B), None, np.inf, B, rule=("ddim", steps, eta), ee_threshold=thr, ee_mode=0)
    grid = _grid(steps)
    n_diff = n_exits = 0
    for k, t in enumerate(grid):
        x = trace["x_in"][t].clone()
        exit_log = torch.full((1000, B), -7, device=dev, dtype=torch.int32)
        score_log = torch.full((1000, 13), -7.0, device=dev)
        smp.run_list(x, [t], [False], noise=nz, exit_log=exit_log, score_log=score_log, use_graph=(k % 2 == 0))
        scores = trace["scores"][t]
        near = ((scores[:-1] - thr).abs() < PROBE_MARGIN_HOT).any(0)
        same = exit_log[t].long() == r_idx[t].long().to(dev)
        assert bool((same | near).all()), (t, exit_log[t].tolist(), r_idx[t].tolist())
        n_diff += int((~same).sum())
        n_exits += int((r_idx[t] < 13).sum())
        assert (score_log[t].cpu() - r_err[t]).abs().max().item() <= PROBE_MARGIN_HOT, t
        mask = torch.ones(1000, dtype=torch.bool, device=dev)
        mask[t] = False
        assert exit_log[mask].eq(-7).all() and score_log[mask].eq(-7.0).all()
        if k + 1 < len(grid) and bool(same.all()):
            assert rel_l2(x, trace["x_in"][grid[k + 1]]) <= EPS_REL_L2, t
    print(f"teacher-forced DDIM {steps}: {n_diff} index mismatches (all within the margin) over {len(grid)} steps x "
          f"{B} samples; {n_exits} early exits in the oracle's log")
    assert n_exits > 0
    # the oracle's own logs: NaN exactly off the grid
    off = _off_grid(steps)
    assert torch.isnan(r_err[off]).all() and torch.isnan(r_idx[off]).all() and torch.isfinite(r_idx[~off]).all()


# ------------------------------------------------------------------------------------------------ 4. public API
def test_get_samples_api_on_the_grid(dev):
    from duodiff_b200 import eesampler as ES
    net = _ee_net("cifar10", 18, dev)
    B, steps = 3, 20
    kw = dict(seed=4, num_channels=3, sample_height=32, sample_width=32, depth=13, use_ddim=True, ddim_steps=steps)
    samples, err, idx = ES.get_samples(net, B, threshold=0.4, **kw)
    assert samples.shape == (B, 32, 32, 3) and samples.dtype == np.float32 and np.isfinite(samples).all()
    assert err.shape == (1000, 13) and idx.shape == (1000, B)
    assert err.dtype == idx.dtype == torch.float32 and err.device.type == idx.device.type == "cpu"
    off = _off_grid(steps)
    assert torch.isnan(err[off]).all() and torch.isnan(idx[off]).all()
    assert torch.isfinite(err[~off]).all() and torch.isfinite(idx[~off]).all()
    assert float(idx[~off].min()) < 13
    _, _, idx0 = ES.get_samples(net, B, threshold=0.0, **kw)
    assert idx0[~off].eq(13).all() and torch.isnan(idx0[off]).all()
    # the default grid: 50 points
    _, _, idx50 = ES.get_samples(net, B, threshold=0.4, seed=4, num_channels=3, sample_height=32, sample_width=32,
                                 depth=13, use_ddim=True)
    assert int((~torch.isnan(idx50[:, 0])).sum()) == 49


@pytest.mark.parametrize("ctype", ["mlp_probe_per_timestep", "mlp_probe_per_layer_per_timestep", "attention_probe"])
def test_other_probe_types_on_the_grid(dev, ctype):
    """The timestep-indexed probe layouts read the probes of each grid timestep (t from device memory in the graph);
    the attention probe has no timestep.  Compact == simulate; the first grid step's score row against the oracle."""
    from duodiff_b200 import eesampler as ES
    name = "celeba_3"
    cfg = CONFIGS[name]
    net = _ee_net(name, 31, dev, ctype=ctype, hot=2.0 if ctype == "attention_probe" else 4.0, spread=False)
    if ctype == "attention_probe":
        g = torch.Generator().manual_seed(37)
        with torch.no_grad():
            for i in range(cfg["depth"]):
                net.matrix[f"{i}"].q.copy_(torch.randn(net.matrix[f"{i}"].q.shape, generator=g).to(dev))
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    spec = O.UViTSpec.from_params(cfg)
    B, steps = 4, 20
    g = torch.Generator().manual_seed(33)
    x_T = torch.randn(B, 3, 64, 64, generator=g)
    noise = torch.randn(1000, B, 3, 64, 64, generator=g)
    with torch.no_grad():
        _, r_cls, _ = O.ee_forward(sd, spec, x_T.to(dev), torch.full((B,), 999.0, device=dev), None,
                                   classifier_type=ctype)
    r_cls = torch.stack([c.reshape(-1) for c in r_cls])
    thr = float(r_cls.median())
    kw = dict(seed=2, num_channels=3, sample_height=64, sample_width=64, threshold=thr, depth=cfg["depth"],
              noise=noise, x_T=x_T, use_ddim=True, ddim_steps=steps)
    s0, e0, i0 = ES.get_samples(net, B, mode=0, **kw)
    s1, _e1, i1 = ES.get_samples(net, B, mode=1, **kw)
    assert np.array_equal(s0, s1) and _same(i0, i1) and np.isfinite(s0).all()
    off = _off_grid(steps)
    assert torch.isnan(i0[off]).all() and torch.isfinite(e0[~off]).all()
    margin = 3e-2 * (1.0 + r_cls.abs().max().item()) if ctype == "attention_probe" else PROBE_MARGIN_HOT
    assert (e0[999] - r_cls.mean(1).cpu()).abs().max().item() <= margin


@pytest.mark.parametrize("steps,eta", [(50, 0.0), (20, 0.05)])
def test_free_running_never_exit_matches_oracle(dev, steps, eta):
    """Threshold 0.0 (no probe fires): the free-running DDIM trajectory against ee_sample_ddim with identical x_T and
    injected noise, reference-init weights, within the free-running bound of tests/test_gpu_parity.py."""
    from duodiff_b200 import eesampler as ES
    net = _ee_net("cifar10_3", 31, dev, hot=0, spread=False)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    spec = O.UViTSpec.from_params(CONFIGS["cifar10_3"])
    B = 2
    g = torch.Generator().manual_seed(14)
    noise = torch.randn(1000, B, 3, 32, 32, generator=g)
    x_T = torch.randn(B, 3, 32, 32, generator=g)
    out, _err, idx = ES.get_samples(net, B, seed=3, num_channels=3, sample_height=32, sample_width=32, threshold=0.0,
                                    depth=3, noise=noise, x_T=x_T, use_ddim=True, ddim_steps=steps, ddim_eta=eta)
    model = lambda x, t, y: O.ee_forward(sd, spec, x, t, y)  # noqa: E731
    x0, _r_err, r_idx = ee_sample_ddim(model, 0.0, 3, x_T.to(dev), noise.to(dev), steps, eta)
    r = rel_l2(torch.from_numpy(out).to(dev), O.to_samples_nhwc(x0))
    print(f"DDIM {steps} eta {eta}, never exiting: free-running rel-L2 {r:.2e}")
    assert r <= IMG_REL_L2
    assert _same(idx, r_idx)


# ------------------------------------------------------------------------------------------------ 5. sharding
def test_batch_invariance_on_the_grid(dev):
    """Shards (x_T rows + noise_row_offset for the Philox stream) reproduce the whole batch: samples and index log bit
    for bit, the batch-mean score log as the row-weighted mean of the shards' within 1e-5."""
    from duodiff_b200 import eesampler as ES
    net = _ee_net("cifar10", 28, dev)
    G, steps = 6, 20
    g = torch.Generator().manual_seed(29)
    x_T = torch.randn(G, 3, 32, 32, generator=g)
    kw = dict(seed=7, num_channels=3, sample_height=32, sample_width=32, threshold=0.4, depth=13, use_ddim=True,
              ddim_steps=steps, ddim_eta=0.05)
    s, e, i = ES.get_samples(net, G, x_T=x_T, **kw)
    parts = [ES.get_samples(net, hi - lo, x_T=x_T[lo:hi].contiguous(), noise_row_offset=lo, **kw)
             for lo, hi in ((0, 4), (4, 6))]
    assert np.array_equal(s, np.concatenate([p[0] for p in parts]))
    assert _same(i, torch.cat([p[2] for p in parts], dim=1))
    mean = (parts[0][1] * 4 + parts[1][1] * 2) / 6
    off = _off_grid(steps)
    assert torch.isnan(mean[off]).all() and (mean[~off] - e[~off]).abs().max().item() <= 1e-5


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _shard_worker(rank, world, port, out):
    from duodiff_b200 import distributed as D
    from duodiff_b200 import eesampler as ES
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.distributed.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(seconds=300))
    try:
        net = _ee_net("cifar10", 28, torch.device("cuda:0"))
        got = D.get_samples_on_rank0(functools.partial(ES.get_samples, model=net), 5, shape=(3, 32, 32), seed=7,
                                     outputs=D.EESAMPLER_OUTPUTS, num_channels=3, sample_height=32, sample_width=32,
                                     threshold=0.4, depth=13, use_ddim=True, ddim_steps=20)
        if rank == 0:
            torch.save(dict(samples=torch.from_numpy(got[0]), err=got[1], idx=got[2]), out)
    finally:
        torch.distributed.destroy_process_group()


def test_two_gloo_shards_on_one_gpu(dev, tmp_path):
    import torch.multiprocessing as mp

    from duodiff_b200 import eesampler as ES
    out = tmp_path / "sharded.pt"
    mp.spawn(_shard_worker, args=(2, _free_port(), str(out)), nprocs=2, join=True)
    got = torch.load(out)
    net = _ee_net("cifar10", 28, dev)
    s, e, i = ES.get_samples(net, 5, seed=7, num_channels=3, sample_height=32, sample_width=32, threshold=0.4,
                             depth=13, use_ddim=True, ddim_steps=20)
    assert np.array_equal(got["samples"].numpy(), s) and _same(got["idx"], i)
    off = _off_grid(20)
    assert torch.isnan(got["err"][off]).all() and (got["err"][~off] - e[~off]).abs().max().item() <= 1e-5


# ------------------------------------------------------------------------------------------------ 6. command line
def test_eesampler_cli_use_ddim(tmp_path):
    from duodiff_b200 import eesampler as ES
    from tests.test_gpu_cli import _png, _write
    ck, cfg = _write(tmp_path, "ee", CONFIGS["cifar10"], 6, wrap=False, ee=True)
    out = tmp_path / "ee_ddim"
    ES.main(["--checkpoint_path", ck, "--config_path", cfg, "--threshold", "0.45", "--batch_size", "3",
             "--output_folder", str(out), "--seed", "2", "--use_ddim", "--ddim_steps", "20"])
    assert sorted(p.name for p in out.iterdir()) == sorted(
        ["0.png", "1.png", "2.png", "statistics.txt", "error_prediction_by_timestep.pt", "indices_by_timestep.pt"])
    err = torch.load(out / "error_prediction_by_timestep.pt")
    idx = torch.load(out / "indices_by_timestep.pt")
    off = _off_grid(20)
    assert err.shape == (1000, 13) and idx.shape == (1000, 3) and idx.dtype == torch.float32
    assert torch.isnan(err[off]).all() and torch.isnan(idx[off]).all()
    assert torch.isfinite(err[~off]).all() and float(idx[~off].min()) < 13
    assert _png(out / "2.png").shape == (32, 32, 4)


def test_torchrun_eesampler_use_ddim(tmp_path):
    from tests.test_gpu_cli import _write
    from tests.test_gpu_cli_distributed import _first_gpu_only, _run
    ck, cfg = _write(tmp_path, "ee", CONFIGS["cifar10"], 6, wrap=False, ee=True)
    args = ["--checkpoint_path", ck, "--config_path", cfg, "--threshold", "0.45", "--batch_size", "5", "--seed", "2",
            "--use_ddim", "--ddim_steps", "20", "--ddim_eta", "0.05"]
    single, multi = tmp_path / "single", tmp_path / "torchrun2"
    env = _first_gpu_only()
    _run([sys.executable, "eesampler.py", *args, "--output_folder", str(single)], env=env)
    out = _run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2", "eesampler.py",
                *args, "--output_folder", str(multi)], env=env)
    assert "Gathered" in out
    names = sorted(p.name for p in single.iterdir())
    assert names == sorted(p.name for p in multi.iterdir()) and len(names) == 5 + 3
    for name in names:
        if name.endswith(".png"):
            assert (single / name).read_bytes() == (multi / name).read_bytes(), name
    assert _same(torch.load(single / "indices_by_timestep.pt"), torch.load(multi / "indices_by_timestep.pt"))
    e1, e2 = torch.load(single / "error_prediction_by_timestep.pt"), torch.load(multi / "error_prediction_by_timestep.pt")
    off = _off_grid(20)
    assert torch.isnan(e2[off]).all() and (e1[~off] - e2[~off]).abs().max().item() <= 1e-5
