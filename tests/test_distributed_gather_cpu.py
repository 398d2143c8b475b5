"""gloo tests (CPU) of the host logic behind the two command lines under torchrun: sharded sampling whose full result
(samples, --timesteps_save intermediates, early-exit logs) is gathered on rank 0, including ranks with empty shards
whose output rows have a shape other than x_T's (a decoding autoencoder) and a dtype other than float32."""
import os
import socket
from datetime import timedelta

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from duodiff_b200 import distributed as D

DEPTH = 5
SHAPE = (3, 4, 4)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _keyed_noise(seed, t, row, shape):
    """Stand-in for the in-kernel Philox stream: a function of (seed, t, GLOBAL row) only."""
    g = torch.Generator().manual_seed((seed * 1000 + t) * 100003 + row)
    return torch.randn(*shape, generator=g)


def _run(batch_size, seed, x_T, noise_row_offset, y, n_inter=0):
    """A batch-invariant stand-in for the sampling loop: returns x_0 and `n_inter` intermediates, [B,C,H,W]."""
    if x_T is None:  # the single-process draw of sampler.get_samples
        x_T = D.global_x_T(seed, batch_size, SHAPE)
    assert x_T.shape[0] == batch_size
    x, kept = x_T.clone(), []
    for t in range(999, 993, -1):
        z = torch.stack([_keyed_noise(seed, t, noise_row_offset + b, x.shape[1:]) for b in range(batch_size)])
        x = 0.9 * x + 0.1 * z + (0 if y is None else y.view(-1, 1, 1, 1).float() * 1e-3)
        if len(kept) < n_inter and t % 2 == 0:
            kept.append(x.clone())
    return x, kept


def fake_sampler(batch_size, seed, x_T=None, noise_row_offset=0, noise=None, y=None):
    """sampler.get_samples-shaped: (samples [B,H,W,C] numpy f32, [two intermediates])."""
    x, kept = _run(batch_size, seed, x_T, noise_row_offset, y, n_inter=2)
    nhwc = lambda a: a.permute(0, 2, 3, 1).contiguous().numpy()  # noqa: E731
    return nhwc(x), [nhwc(k) for k in kept]


def fake_decoding_sampler(batch_size, seed, x_T=None, noise_row_offset=0, noise=None, y=None):
    """Like fake_sampler, but the rows come back "decoded" to [2H, 2W, 2] float64, as an autoencoder changes them."""
    x, kept = _run(batch_size, seed, x_T, noise_row_offset, y, n_inter=1)

    def decode(a):
        img = a[:, :2].repeat_interleave(2, 2).repeat_interleave(2, 3)
        return img.permute(0, 2, 3, 1).contiguous().double().numpy()
    return decode(x), [decode(k) for k in kept]


def fake_eesampler(batch_size, seed, x_T=None, noise_row_offset=0, noise=None, y=None, decode=False):
    """eesampler.get_samples-shaped: (samples, error log [1000, depth] = batch mean, index log [1000, B] float32)."""
    x, _ = _run(batch_size, seed, x_T, noise_row_offset, y)
    rows = x.flatten(1)
    per_row = torch.stack([rows[:, :DEPTH].sin().abs() + 1e-4 * t for t in range(1000)])  # [1000, B, depth]
    idx = (rows[:, 0].abs() * 7).floor().clamp(max=DEPTH).view(1, -1) + torch.zeros(1000, 1)
    samples = x.permute(0, 2, 3, 1).contiguous().numpy()
    if decode:
        samples = np.repeat(samples[..., :1], 3, axis=1).astype(np.float64)
    return samples, per_row.mean(1), idx.to(torch.float32)


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    # a short timeout turns a hang of a mismatched collective into an error
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(seconds=60))


def _assert_same(got, ref):
    assert type(got) is type(ref)
    if isinstance(ref, (tuple, list)):
        assert len(got) == len(ref)
        for a, b in zip(got, ref):
            _assert_same(a, b)
    elif isinstance(ref, np.ndarray):
        assert got.dtype == ref.dtype and got.shape == ref.shape and np.array_equal(got, ref)
    else:
        assert got.dtype == ref.dtype and torch.equal(got, ref)


def _check_ee(got, ref):
    assert np.array_equal(got[0], ref[0]) and got[0].dtype == ref[0].dtype
    assert torch.equal(got[2], ref[2]), "index log not gathered along the batch axis in rank order"
    assert got[1].dtype == ref[1].dtype and got[1].shape == ref[1].shape
    assert not torch.isnan(got[1]).any()
    assert (got[1] - ref[1]).abs().max().item() <= 1e-6


def _worker_uneven(rank, world, port, G, flag):
    _init(rank, world, port)
    try:
        y = torch.arange(G)
        # sampler-shaped: samples + two intermediates, uneven shards (4 + 3)
        got = D.get_samples_on_rank0(fake_sampler, G, shape=SHAPE, seed=5, y=y)
        # eesampler-shaped: index log along axis 1, error log as a row-weighted mean
        got_ee = D.get_samples_on_rank0(fake_eesampler, G, shape=SHAPE, seed=2, outputs=D.EESAMPLER_OUTPUTS)
        if rank == 0:
            _assert_same(got, fake_sampler(G, 5, y=y))
            assert len(got[1]) == 2
            _check_ee(got_ee, fake_eesampler(G, 2))
            open(flag, "w").write("ok")
        else:
            assert got is None and got_ee is None
    finally:
        dist.destroy_process_group()


def test_two_ranks_gather_full_result_on_rank0(tmp_path):
    flag = tmp_path / "ok"
    mp.spawn(_worker_uneven, args=(2, _free_port(), 7, str(flag)), nprocs=2, join=True)
    assert flag.read_text() == "ok"


def _worker_empty(rank, world, port, G, flag):
    _init(rank, world, port)
    try:
        lo, hi = D.shard_bounds(G, rank, world)
        calls = []

        def counted(fn):
            def f(**kw):
                calls.append(kw["batch_size"])
                return fn(**kw)
            return f
        got = D.get_samples_on_rank0(counted(fake_decoding_sampler), G, shape=SHAPE, seed=3)
        got_ee = D.get_samples_on_rank0(counted(lambda **kw: fake_eesampler(decode=True, **kw)), G, shape=SHAPE,
                                        seed=4, outputs=D.EESAMPLER_OUTPUTS)
        assert calls == ([hi - lo] * 2 if hi > lo else []), "an empty shard must not run the sampler"
        if rank == 0:
            ref = fake_decoding_sampler(G, 3)
            assert ref[0].shape[1:] == (8, 8, 2) and ref[0].dtype == np.float64
            _assert_same(got, ref)
            _check_ee(got_ee, fake_eesampler(G, 4, decode=True))
            open(flag, "w").write("ok")
        else:
            assert got is None and got_ee is None
    finally:
        dist.destroy_process_group()


def test_empty_shard_with_decoded_float64_rows(tmp_path):
    """3 ranks, 2 images: rank 2 has no rows, runs nothing, and still joins every collective."""
    flag = tmp_path / "ok"
    mp.spawn(_worker_empty, args=(3, _free_port(), 2, str(flag)), nprocs=3, join=True)
    assert flag.read_text() == "ok"


def _worker_sharded_decode(rank, world, port, G, flag):
    _init(rank, world, port)
    try:
        got = D.get_samples_sharded(fake_decoding_sampler, G, shape=SHAPE, seed=6)
        ref = torch.from_numpy(fake_decoding_sampler(G, 6)[0])
        assert got.dtype == ref.dtype and torch.equal(got, ref)
        if rank == 0:
            open(flag, "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_get_samples_sharded_empty_shard_with_decoded_rows(tmp_path):
    """The all-gathering get_samples_sharded: an empty shard's zero rows take the decoded row shape and dtype."""
    flag = tmp_path / "ok"
    mp.spawn(_worker_sharded_decode, args=(3, _free_port(), 2, str(flag)), nprocs=3, join=True)
    assert flag.read_text() == "ok"


def test_single_process_is_the_plain_call(monkeypatch):
    """Without a process group the sampler runs once on the whole batch, with no x_T handed in."""
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    seen = []

    def fn(**kw):
        seen.append(kw)
        return fake_sampler(**kw)
    got = D.get_samples_on_rank0(fn, 3, shape=SHAPE, seed=1)
    _assert_same(got, fake_sampler(3, 1))
    assert seen == [dict(batch_size=3, seed=1, noise=None, y=None)]
    with D.cli_process_group() as (rank, world, device):
        assert (rank, world, device) == (0, 1, torch.device("cuda:0")) and not dist.is_initialized()


@pytest.mark.parametrize("G,world", [(7, 2), (2, 3), (1, 8), (128, 8)])
def test_every_row_has_one_owner(G, world):
    spans = [D.shard_bounds(G, r, world) for r in range(world)]
    assert spans[0][1] > spans[0][0], "rank 0 always has rows: the empty ranks take shapes from it"
    assert sum(hi - lo for lo, hi in spans) == G
