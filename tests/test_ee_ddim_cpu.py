"""CPU tests of DDIM sampling with early exit: the `eesampler.py --use_ddim` flags, the argument checks of
eesampler.get_samples, the early-exit DDIM oracle against the plain DDIM oracle, the C ABI of
ddb_sampler_run_list_logs, and the gather of NaN (off-grid) log rows over two gloo ranks."""
import math
import os
import socket
from datetime import timedelta

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from duodiff_b200 import _lib
from duodiff_b200 import distributed as D
from duodiff_b200 import eesampler as ES
from duodiff_b200.configs import CONFIGS
from duodiff_b200.ddpm import ddim_timesteps
from oracle import uvit_oracle as O
from oracle.ee_ddim_oracle import ee_sample_ddim

torch.set_num_threads(4)


# ------------------------------------------------------------------------------------------------ command line
def _base_argv():
    return ["--threshold", "0.1", "--checkpoint_path", "a.pth", "--batch_size", "4", "--output_folder", "o",
            "--config_path", "c.yaml"]


def test_ddim_flags_are_absent_unless_given():
    a = ES.get_args(_base_argv())
    assert sorted(vars(a)) == sorted(["seed", "threshold", "checkpoint_path", "batch_size", "output_folder",
                                      "config_path", "class_id"])
    a = ES.get_args(_base_argv() + ["--use_ddim"])
    assert a.use_ddim is True and not hasattr(a, "ddim_steps") and not hasattr(a, "ddim_eta")
    a = ES.get_args(_base_argv() + ["--use_ddim", "--ddim_steps", "20", "--ddim_eta", "0.5"])
    assert (a.use_ddim, a.ddim_steps, a.ddim_eta) == (True, 20, 0.5)


@pytest.mark.parametrize("extra", [["--ddim_steps", "20"], ["--ddim_eta", "1.0"], ["--use_ddim", "--ddim_steps", "1"]])
def test_ddim_flag_errors(extra):
    with pytest.raises(SystemExit):
        ES.get_args(_base_argv() + extra)


# ------------------------------------------------------------------------------------------------ get_samples
def _small_ee():
    import duodiff_b200 as ddb
    params = dict(CONFIGS["cifar10_3"], embed_dim=64, num_heads=2)
    torch.manual_seed(0)
    return ddb.EarlyExitUViT(ddb.UViT(**params), "mlp_probe_per_layer").eval(), params


def test_get_samples_rejects_bad_ddim_arguments():
    net, _ = _small_ee()
    kw = dict(batch_size=2, seed=0, num_channels=3, sample_height=32, sample_width=32, threshold=0.1, depth=3)
    for bad in (dict(ddim_steps=20), dict(ddim_eta=0.0), dict(ddim_steps=50, ddim_eta=1.0)):
        with pytest.raises(ValueError, match="use_ddim"):
            ES.get_samples(net, **kw, **bad)
    for n in (0, 1):
        with pytest.raises(ValueError, match="at least 2"):
            ES.get_samples(net, **kw, use_ddim=True, ddim_steps=n)
    with pytest.raises(ValueError, match="strictly decreasing"):  # more grid points than timesteps
        ES.get_samples(net, **kw, use_ddim=True, ddim_steps=1001)


# ------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("steps,eta", [(6, 0.0), (5, 0.01)])
def test_oracle_never_exiting_is_plain_ddim(steps, eta):
    """Threshold 0.0: no sigmoid probe is <= 0, every sample takes the final head, and the early-exit DDIM loop is
    uvit_oracle.sample_ddim on the backbone.  (eta stays small: the reference's last step, s = 0, takes
    sqrt(1 - abar_0 - eta * beta_tilde_t), which is negative on these coarse grids from eta = 0.05 on.)"""
    net, params = _small_ee()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    spec = O.UViTSpec.from_params(params)
    g = torch.Generator().manual_seed(1)
    x_T = torch.randn(2, 3, 32, 32, generator=g)
    noise = torch.randn(1000, 2, 3, 32, 32, generator=g)
    trace = {}
    x_ee, err, idx = ee_sample_ddim(lambda x, t, y: O.ee_forward(sd, spec, x, t, y), 0.0, spec.depth, x_T.clone(),
                                    noise, steps, eta, trace=trace)
    x_ref = O.sample_ddim(lambda x, t, y: O.uvit_forward(sd, spec, x, t, y, pfx="uvit."), None, math.inf, x_T.clone(),
                          noise, steps, eta)
    assert float((x_ee - x_ref).norm() / x_ref.norm()) <= 1e-6
    grid = ddim_timesteps(steps)[:-1]
    assert sorted(trace["x_in"]) == sorted(grid)
    off = torch.ones(1000, dtype=torch.bool)
    off[grid] = False
    assert err.shape == (1000, spec.depth) and idx.shape == (1000, 2)
    assert torch.isnan(err[off]).all() and torch.isnan(idx[off]).all()
    assert torch.isfinite(err[grid]).all() and idx[grid].eq(spec.depth).all()


# ------------------------------------------------------------------------------------------------ C ABI
def test_run_list_logs_in_the_exported_abi():
    from pathlib import Path

    from duodiff_b200 import _build
    res, args = _lib._SIGS["ddb_sampler_run_list_logs"]
    assert res is _lib.C.c_int and len(args) == 14
    assert args[:10] == _lib._SIGS["ddb_sampler_run_list"][1][:10]  # the arguments of ddb_sampler_run_list first
    _build.build()
    lib = _lib.load()
    assert "ddb_sampler_run_list_logs" in _lib.EXPORTED_SYMBOLS and hasattr(lib, "ddb_sampler_run_list_logs")
    assert lib.ddb_sampler_run_list_logs.argtypes == args
    header = (Path(__file__).resolve().parents[1] / "include" / "duodiff_b200.h").read_text()
    assert "int ddb_sampler_run_list_logs(" in header


# ------------------------------------------------------------------------------------------------ sharding
DEPTH, G = 4, 5
GRID = ddim_timesteps(20)[:-1]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _logs(lo, hi):
    """A shard's (samples, error log, index log) as eesampler.get_samples(use_ddim=True) returns them: NaN rows off
    the grid.  The error log rows are the same on every shard, so the weighted mean is exact."""
    off = torch.ones(1000, dtype=torch.bool)
    off[GRID] = False
    err = torch.arange(1000 * DEPTH, dtype=torch.float32).view(1000, DEPTH) / 7
    idx = (torch.arange(1000).view(-1, 1) + torch.arange(lo, hi).view(1, -1)).remainder(DEPTH + 1).float()
    err[off], idx[off] = float("nan"), float("nan")
    samples = np.arange(lo, hi, dtype=np.float32).reshape(-1, 1, 1, 1) * np.ones((1, 2, 2, 3), np.float32)
    return samples, err, idx


def _worker(rank, world, port, flag):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(seconds=60))
    try:
        lo, hi = D.shard_bounds(G, rank, world)
        got = D.gather_to_rank0(_logs(lo, hi) if hi > lo else None, G, D.EESAMPLER_OUTPUTS)
        if rank == 0:
            ref = _logs(0, G)
            assert np.array_equal(got[0], ref[0])
            for a, b in zip(got[1:], ref[1:]):
                assert a.dtype == b.dtype == torch.float32 and a.shape == b.shape
                assert torch.equal(torch.isnan(a), torch.isnan(b)) and torch.isnan(a).sum() > 0
                assert torch.equal(a[GRID], b[GRID])
            open(flag, "w").write("ok")
        else:
            assert got is None
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 6])
def test_gather_keeps_off_grid_rows_nan(tmp_path, world):
    """2 ranks (3 + 2 samples) and 6 ranks (one of them with an empty shard, whose zeros carry weight 0)."""
    flag = tmp_path / "ok"
    mp.spawn(_worker, args=(world, _free_port(), str(flag)), nprocs=world, join=True)
    assert flag.read_text() == "ok"
