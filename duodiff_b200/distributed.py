"""Data-parallel sharding of the sample batch (SURVEY.md §8e): one process per GPU, no collective inside the loop,
one gather of the finished samples at the end (plus the early-exit logs).  Works over NCCL (GPU) and gloo (the two
command lines, which gather host arrays, and the CPU tests of the host logic)."""
from __future__ import annotations

import contextlib
import os

import numpy as np
import torch
import torch.distributed as dist


def env_rank_world():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))


def _rank_world():
    return (dist.get_rank(), dist.get_world_size()) if dist.is_available() and dist.is_initialized() else (0, 1)


@contextlib.contextmanager
def cli_process_group():
    """Process set-up of `python sampler.py …` / `eesampler.py …`, alone or under `torchrun --nproc-per-node N`.

    Yields (rank, world, device).  With WORLD_SIZE unset or 1 it does nothing and the device is cuda:0.  Otherwise it
    binds the process to cuda:(LOCAL_RANK % device_count) -- before any model or autoencoder is built, since those
    allocate on the current device -- and joins a gloo process group (torchrun's env:// rendezvous), destroyed when
    the block ends, on success or on error.  gloo because the one collective moves host arrays (get_samples returns
    numpy samples and CPU logs), and because it lets several ranks share one GPU, which NCCL refuses."""
    rank, world, local_rank = env_rank_world()
    if world <= 1:
        yield 0, 1, torch.device("cuda:0")
        return
    device = torch.device("cuda", local_rank % torch.cuda.device_count())
    torch.cuda.set_device(device)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        yield rank, world, device
    finally:
        dist.destroy_process_group()


def barrier() -> None:
    """dist.barrier() when a process group is up, else nothing."""
    if _rank_world()[1] > 1:
        dist.barrier()


def shard_bounds(global_batch: int, rank: int, world: int):
    """Rows [lo, hi) of the global batch owned by `rank`: contiguous, sizes differ by at most one."""
    base, rem = divmod(global_batch, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_gather_rows(local: torch.Tensor, global_rows: int) -> torch.Tensor:
    """Concatenate per-rank row blocks (possibly uneven) in rank order on every rank."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local
    world = dist.get_world_size()
    sizes = [shard_bounds(global_rows, r, world) for r in range(world)]
    max_rows = max(hi - lo for lo, hi in sizes)
    pad = torch.zeros((max_rows, *local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    bufs = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(bufs, pad)
    return torch.cat([b[: hi - lo] for b, (lo, hi) in zip(bufs, sizes)], dim=0)


def all_reduce_weighted_mean(local_mean: torch.Tensor, local_rows: int, global_rows: int) -> torch.Tensor:
    """Batch-mean logs (eesampler.py:71) of the shards -> the mean over the global batch."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local_mean
    acc = local_mean * float(local_rows)
    dist.all_reduce(acc, op=dist.ReduceOp.SUM)
    return acc / float(global_rows)


def global_x_T(seed: int, global_batch: int, shape) -> torch.Tensor:
    """The initial noise of the whole global batch, drawn like the reference's single process does (sampler.py:99-100:
    seed_everything(seed), then one CPU randn of the full batch).  Every rank draws the same tensor and keeps its rows."""
    from ._io import seed_everything
    seed_everything(seed)
    return torch.randn(global_batch, *shape)


def get_samples_sharded(get_samples_fn, global_batch: int, *, shape=None, noise=None, y=None, seed: int = 0,
                        x_T=None, **kw):
    """Run `sampler.get_samples`-like `get_samples_fn(batch_size=..., seed=..., x_T=..., noise_row_offset=..., noise=...,
    y=...)` on this rank's shard of a global batch and gather the finished samples on every rank.

    The result is the single-process result of `get_samples(batch_size=global_batch, seed=seed)` row for row, whatever
    the world size: every rank draws the global x_T (`shape` = [C,H,W]; or is handed `x_T` [G,C,H,W]) and keeps rows
    [lo, hi); the per-step noise is either injected (`noise` [1000,G,C,H,W]) or the in-kernel Philox stream keyed by
    (seed, t, global element index) through `noise_row_offset=lo`; the kernels are batch-invariant.  So a caller
    looping over seeds gets the same, disjoint sample sets as on one GPU (no `seed + rank` collisions).  A rank whose
    shard is empty (world > global_batch) skips the computation and contributes no rows."""
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist.is_initialized() else (0, 1)
    lo, hi = shard_bounds(global_batch, rank, world)
    if x_T is None:
        if shape is None:
            raise ValueError("get_samples_sharded needs shape=[C,H,W] (to draw the global x_T) or x_T")
        x_T = global_x_T(seed, global_batch, tuple(shape))
    x_T = torch.as_tensor(x_T)
    use_cuda = dist.is_initialized() and dist.get_backend() == "nccl"
    t = None
    if hi > lo:
        n_local = noise[:, lo:hi].contiguous() if noise is not None else None
        y_local = y[lo:hi].contiguous() if y is not None else None
        out = get_samples_fn(batch_size=hi - lo, seed=seed, x_T=x_T[lo:hi].contiguous(), noise_row_offset=lo,
                             noise=n_local, y=y_local, **kw)
        samples = out[0] if isinstance(out, tuple) else out
        t = torch.as_tensor(samples)
    if world > global_batch:
        # some shard is empty: its zero rows take their shape and dtype from rank 0 (which always has rows), not from
        # x_T -- with an autoencoder the samples are decoded images, not latents
        row_shape, dtype = _from_rank0((tuple(t.shape[1:]), t.dtype) if rank == 0 else None)
        if t is None:
            t = torch.zeros((0, *row_shape), dtype=dtype)
    if use_cuda:
        t = t.cuda()
    return all_gather_rows(t, global_batch)


def _from_rank0(obj):
    """Rank 0's `obj` (any picklable value) on every rank."""
    box = [obj]
    dist.broadcast_object_list(box, src=0)
    return box[0]


# How get_samples_on_rank0 combines each element of a get_samples-like result tuple over the shards
ROWS = "rows"            # per-row array, batch axis 0: gathered in rank order
ROWS_LIST = "rows_list"  # list of such arrays (the --timesteps_save intermediates)
COLS = "cols"            # per-row array, batch axis 1 (indices_by_timestep [1000, B])
MEAN = "mean"            # batch mean (error_prediction_by_timestep [1000, depth]): row-count-weighted mean
SAMPLER_OUTPUTS = (ROWS, ROWS_LIST)          # sampler.get_samples -> (samples, [intermediates])
EESAMPLER_OUTPUTS = (ROWS, MEAN, COLS)       # eesampler.get_samples -> (samples, error log, index log)


def run_shard(get_samples_fn, global_batch: int, *, shape, seed: int = 0, noise=None, y=None, **kw):
    """This rank's part of `get_samples_fn(batch_size=global_batch, seed=seed, ...)`: the call itself without a
    process group (world 1); otherwise the call on rows [lo, hi) with x_T = those rows of `global_x_T(seed,
    global_batch, shape)` and `noise_row_offset=lo` (see get_samples_sharded), or None if the shard is empty -- then
    `get_samples_fn` is not called, so the rank needs no model."""
    rank, world = _rank_world()
    if world == 1:
        return get_samples_fn(batch_size=global_batch, seed=seed, noise=noise, y=y, **kw)
    lo, hi = shard_bounds(global_batch, rank, world)
    if hi == lo:
        return None
    x_T = global_x_T(seed, global_batch, tuple(shape))
    return get_samples_fn(batch_size=hi - lo, seed=seed, x_T=x_T[lo:hi].contiguous(), noise_row_offset=lo,
                          noise=noise[:, lo:hi].contiguous() if noise is not None else None,
                          y=y[lo:hi].contiguous() if y is not None else None, **kw)


def gather_to_rank0(local, global_batch: int, outputs=SAMPLER_OUTPUTS):
    """Combine the per-rank results of `run_shard` into the single-process result, on rank 0 only (None elsewhere).

    `outputs` says how each element of the result tuple combines (ROWS, ROWS_LIST, COLS, MEAN).  Per-row arrays are
    padded to the largest shard and gathered -- not all-gathered: decoded ImageNet-256 samples of a large batch would
    otherwise be copied to every rank.  Numpy arrays stay numpy arrays, tensors stay CPU tensors.  A rank with an
    empty shard (`local` None) takes every element's shape and dtype from rank 0, which always has rows, and adds
    weight 0 to the means.  Without a process group `local` is returned as is."""
    rank, world = _rank_world()
    if world == 1:
        return local
    lo, hi = shard_bounds(global_batch, rank, world)

    def describe(v):
        return (isinstance(v, np.ndarray), torch.as_tensor(v).dtype, tuple(v.shape))
    meta = _from_rank0([[describe(v) for v in x] if kind == ROWS_LIST else describe(x)
                        for kind, x in zip(outputs, local)] if rank == 0 else None)

    def combine(kind, v, desc):
        is_np, dtype, shape = desc
        if v is None:  # empty shard
            axis = {ROWS: 0, COLS: 1}.get(kind)
            v = torch.zeros(shape[:axis] + (0,) + shape[axis + 1:] if axis is not None else shape, dtype=dtype)
        v = torch.as_tensor(v).cpu()
        if kind == MEAN:
            acc = v.double() * (hi - lo)  # an empty shard's zeros: weight 0, and no NaN from an empty mean
            dist.reduce(acc, dst=0, op=dist.ReduceOp.SUM)
            out = (acc / global_batch).to(dtype)
        else:
            out = _gather_rows_to_rank0(v, global_batch, axis=1 if kind == COLS else 0)
        if rank != 0:
            return None
        return out.numpy() if is_np else out

    result = []
    for i, kind in enumerate(outputs):
        x = local[i] if local is not None else None
        if kind == ROWS_LIST:
            result.append([combine(ROWS, x[j] if x is not None else None, d) for j, d in enumerate(meta[i])])
        else:
            result.append(combine(kind, x, meta[i]))
    return tuple(result) if rank == 0 else None


def get_samples_on_rank0(get_samples_fn, global_batch: int, *, shape, seed: int = 0, outputs=SAMPLER_OUTPUTS,
                         noise=None, y=None, **kw):
    """`get_samples_fn(batch_size=global_batch, seed=seed, ...)`'s result on rank 0, computed by all ranks of the
    process group, each on its shard: (samples, [intermediates]) for sampler.get_samples (`outputs` =
    SAMPLER_OUTPUTS), (samples, error_prediction_by_timestep, indices_by_timestep) for eesampler.get_samples
    (EESAMPLER_OUTPUTS).  None on the other ranks.  Samples, intermediates and index logs equal the single-process
    ones row for row (the kernels are batch-invariant); the error log is a weighted mean of the shards' means, so it
    differs from the single-process one in the last bits.  `shape` = [C,H,W] of x_T."""
    local = run_shard(get_samples_fn, global_batch, shape=shape, seed=seed, noise=noise, y=y, **kw)
    return gather_to_rank0(local, global_batch, outputs)


def _gather_rows_to_rank0(local: torch.Tensor, global_rows: int, axis: int = 0):
    """Concatenate per-rank blocks (possibly uneven, possibly empty) along `axis` in rank order, on rank 0 only."""
    rank, world = _rank_world()
    sizes = [shard_bounds(global_rows, r, world) for r in range(world)]
    rows = local.movedim(axis, 0)
    pad = torch.zeros((max(hi - lo for lo, hi in sizes), *rows.shape[1:]), dtype=rows.dtype)
    pad[: rows.shape[0]] = rows
    bufs = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
    dist.gather(pad, bufs, dst=0)
    if rank != 0:
        return None
    return torch.cat([b[: hi - lo] for b, (lo, hi) in zip(bufs, sizes)], dim=0).movedim(0, axis).contiguous()


def gather_ee_logs(error_prediction_local: torch.Tensor, indices_local: torch.Tensor, global_rows: int):
    """eesampler logs of the shards -> the logs of the global batch (eesampler.py:54-55,71-72):
    ``indices_by_timestep`` [1000, B_local] is gathered along the batch axis in rank order, and
    ``error_prediction_by_timestep`` [1000, depth] (a batch mean) is combined as a row-count-weighted mean."""
    local_rows = indices_local.shape[1]
    idx = all_gather_rows(indices_local.t().contiguous(), global_rows).t().contiguous()
    err = all_reduce_weighted_mean(error_prediction_local, local_rows, global_rows)
    return err, idx
