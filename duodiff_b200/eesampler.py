"""Drop-in for the reference's ``eesampler.py`` (DeeDiff / AdaDiff early-exit sampling): same ``get_samples``
signature, logs and CLI flags (eesampler.py:40-89,114-134).  The loop runs inside libduodiff_b200.so.

    python -m duodiff_b200.eesampler --checkpoint_path ee.pth --config_path configs/deediff_celeba.yaml \
        --threshold 0.08 --batch_size 128 --output_folder out/
"""
from __future__ import annotations

import functools
import time
from argparse import SUPPRESS, ArgumentParser
from pathlib import Path

import numpy as np
import torch

from . import _io
from . import distributed as D
from .autoencoder import get_autoencoder
from .ddpm import cached_sampler
from .sampler import _ddim_plan, _pick_device, draw_labels
from .early_exit import EarlyExitUViT
from .uvit import UViT


def get_samples(model, batch_size: int, seed: int, num_channels: int, sample_height: int, sample_width: int,
                threshold: float, depth: int, y=None, autoencoder=None, *, noise=None, mode: int = 0,
                use_graph: bool = True, device=None, x_T=None, noise_row_offset: int = 0, use_ddim: bool = False,
                ddim_steps=None, ddim_eta=None):
    """eesampler.py:40-89 -> (samples [B,H,W,C] numpy, error_prediction_by_timestep [1000,depth],
    indices_by_timestep [1000,B]) with both logs as CPU float32 tensors indexed by t like the reference's.

    ``mode`` 0 evaluates every probe and head like the reference ("simulate"); ``mode`` 1 really skips the layers after
    a sample's exit ("compact"): samples and ``indices_by_timestep`` are bit-identical to mode 0, but row t of
    ``error_prediction_by_timestep`` then holds, per layer, the mean probe output over the samples STILL IN THE BATCH at
    that layer (NaN once the batch is empty) -- the reference's mean over the whole batch (eesampler.py:71) would need
    the skipped layers.  Any ``threshold`` is legal; a negative one selects layer 0's head for every sample, as the
    reference's argmax over an all-false mask does.  ``x_T`` / ``noise_row_offset``: see sampler.get_samples.

    DDIM (not in the reference's eesampler.py): ``use_ddim`` walks the strided grid of ``sampler.get_samples(use_ddim=
    True)`` -- ``ddim_steps`` points (default 50), ``ddim_steps - 1`` model evaluations, the update of sampler.py:110-120
    with its sigma_t^2 * z noise term scaled by ``ddim_eta`` (default 0) -- with the same early exit at every step.  The
    logs keep their shapes and dtypes; rows of timesteps the grid does not visit are NaN in both (a row of zeros would
    read as "every sample left at layer 0").  ``ddim_steps`` / ``ddim_eta`` without ``use_ddim`` raise ValueError."""
    steps = flags = None
    if use_ddim:
        ddim_steps = 50 if ddim_steps is None else int(ddim_steps)
        ddim_eta = 0.0 if ddim_eta is None else float(ddim_eta)
        if ddim_steps < 2:
            raise ValueError(f"ddim_steps={ddim_steps}: the grid needs at least 2 points (one model evaluation)")
        steps, flags = _ddim_plan(ddim_steps, False, np.inf)
    elif ddim_steps is not None or ddim_eta is not None:
        raise ValueError("ddim_steps / ddim_eta select the DDIM grid: they need use_ddim=True")
    dev = _pick_device(model, device)
    _io.seed_everything(seed)
    if x_T is None:
        x = torch.randn(batch_size, num_channels, sample_height, sample_width)
    else:
        x = torch.as_tensor(x_T, dtype=torch.float32).detach().cpu().contiguous()
        if tuple(x.shape) != (batch_size, num_channels, sample_height, sample_width):
            raise ValueError(f"x_T has shape {tuple(x.shape)}")
    x = x.pin_memory().to(dev, non_blocking=True)
    with torch.cuda.device(dev):
        eng = model.engine(batch_size)
        rule = ("ddim", ddim_steps, ddim_eta) if use_ddim else "predict_noise"
        sampler = cached_sampler(eng, None, np.inf, batch_size, rule=rule, ee_threshold=threshold, ee_mode=mode)
        sampler.set_noise_offset(noise_row_offset)
        exit_log = torch.zeros(1000, batch_size, device=dev, dtype=torch.int32)
        score_log = torch.zeros(1000, depth, device=dev, dtype=torch.float32)
        if noise is not None:
            noise = noise.to(device=dev, dtype=torch.float32).contiguous()
        if use_ddim:
            sampler.run_list(x, steps, flags, y=y, noise=noise, seed=seed, exit_log=exit_log, score_log=score_log,
                             use_graph=use_graph)
        else:
            sampler.run(x, y=y, noise=noise, seed=seed, exit_log=exit_log, score_log=score_log, use_graph=use_graph)
        if autoencoder:  # eesampler.py:84-85
            x = autoencoder.decode(x).contiguous()
        samples = sampler.finalize(x).cpu().numpy()
    score_log, exit_log = score_log.cpu(), exit_log.cpu().to(torch.float32)
    if use_ddim:
        off_grid = torch.ones(1000, dtype=torch.bool)
        off_grid[steps] = False
        score_log[off_grid] = float("nan")
        exit_log[off_grid] = float("nan")
    return samples, score_log, exit_log


def dump_samples(samples, output_folder: Path):
    """eesampler.py:92-99 — per-sample PNGs, clipped to [0,1]."""
    for i, s in enumerate(samples):
        _io._save_png(Path(output_folder) / f"{i}.png", np.clip(s, 0, 1))


def dump_statistics(elapsed_time, error_prediction_by_timestep, indices_by_timestep, output_folder: Path):
    """eesampler.py:102-111."""
    output_folder = Path(output_folder)
    with open(output_folder / "statistics.txt", "w") as f:
        f.write(f"Elapsed time: {elapsed_time} s\n")
    torch.save(error_prediction_by_timestep, output_folder / "error_prediction_by_timestep.pt")
    torch.save(indices_by_timestep, output_folder / "indices_by_timestep.pt")


def get_args(argv=None):
    p = ArgumentParser()
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--threshold", type=float, required=True)
    p.add_argument("--checkpoint_path", type=str, required=True)
    p.add_argument("--batch_size", type=int, required=True)
    p.add_argument("--output_folder", type=str, required=True)
    p.add_argument("--config_path", type=str, required=True, help="Path to yaml config file")
    p.add_argument("--class_id", type=int, default=None, help="Number up to 1000 that corresponds to a class")
    # not flags of the reference's eesampler.py: absent from the namespace unless given, so DDPM runs parse as before
    p.add_argument("--use_ddim", action="store_true", default=SUPPRESS,
                   help="Sample on the strided DDIM grid of sampler.py --use_ddim, with early exit at every step")
    p.add_argument("--ddim_steps", type=int, default=SUPPRESS, help="DDIM grid points (default 50; needs --use_ddim)")
    p.add_argument("--ddim_eta", type=float, default=SUPPRESS, help="DDIM eta (default 0; needs --use_ddim)")
    args = p.parse_args(argv)
    if not getattr(args, "use_ddim", False):
        for flag in ("ddim_steps", "ddim_eta"):
            if hasattr(args, flag):
                p.error(f"--{flag} needs --use_ddim")
    elif getattr(args, "ddim_steps", 2) < 2:
        p.error("--ddim_steps needs at least 2 grid points (one model evaluation)")
    return args


def main(argv=None):
    """The reference's CLI.  Under `torchrun --nproc-per-node N` each rank samples its shard of the --batch_size
    images (duodiff_b200.distributed) and rank 0 writes exactly the files a single process writes."""
    args = get_args(argv)
    out_dir = Path(args.output_folder)
    if D.env_rank_world()[0] == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
    if not torch.cuda.is_available():
        raise RuntimeError("duodiff_b200.eesampler needs a B200 (sm_100) GPU; there is no CPU path")
    with D.cli_process_group() as (rank, world, device):
        print(f"Using device {device}")
        cfg = _io.load_config(args.config_path)
        mp = cfg["model_params"]
        lo, hi = D.shard_bounds(args.batch_size, rank, world)
        model = autoencoder = None
        if hi > lo:  # a rank with an empty shard (more ranks than images) builds nothing
            model = EarlyExitUViT(UViT(**_io.uvit_kwargs(cfg), max_batch=hi - lo), mp["classifier_type"])
            _io.load_checkpoint_into(model, args.checkpoint_path)
            model = model.eval().to(device)
        _io.seed_everything(args.seed)
        y = None
        if args.class_id is not None:
            y = draw_labels(args.batch_size, mp.get("num_classes", -1)).to(device)
        if "autoencoder" in cfg and hi > lo:  # eesampler.py:184-189
            autoencoder = get_autoencoder(cfg["autoencoder"]["autoencoder_checkpoint_path"])
        extra = {k: getattr(args, k) for k in ("use_ddim", "ddim_steps", "ddim_eta") if hasattr(args, k)}
        D.barrier()  # every rank has loaded its model: the clock starts together
        tic = time.time()
        local = D.run_shard(
            functools.partial(get_samples, model=model), args.batch_size,
            shape=(mp["in_chans"], mp["img_size"], mp["img_size"]), seed=args.seed, y=y,
            num_channels=mp["in_chans"], sample_height=mp["img_size"], sample_width=mp["img_size"],
            threshold=args.threshold, depth=mp["depth"], autoencoder=autoencoder, **extra)
        D.barrier()  # every shard is done: what follows is the gather alone
        t_gather = time.time()
        result = D.gather_to_rank0(local, args.batch_size, D.EESAMPLER_OUTPUTS)
        tac = time.time()
        if rank != 0:
            return
        if world > 1:
            print(f"Gathered {args.batch_size} samples from {world} ranks in {tac - t_gather:.3f} s")
        samples, err_log, idx_log = result
        dump_statistics(tac - tic, err_log, idx_log, out_dir)
        dump_samples(samples, out_dir)


if __name__ == "__main__":
    main()
