"""Drop-in for the reference's ``sampler.py``: same ``get_samples`` signature and CLI flags (sampler.py:82-155,192-252),
but the 1000-step loop — U-ViT forwards, the DuoDiff hand-off after ``t == 1000 - t_switch`` and the per-step DDPM
update — runs inside libduodiff_b200.so as CUDA-graph replays of hand-written sm_100a kernels.

    python -m duodiff_b200.sampler --checkpoint_path early.pth --config_path configs/uvit_celeba_3.yaml \
        --checkpoint_path_late full.pth --config_path_late configs/uvit_celeba.yaml --t_switch 300 \
        --batch_size 128 --parametrization predict_noise --output_folder out/
"""
from __future__ import annotations

import functools
import time
from argparse import ArgumentParser
from pathlib import Path
from typing import List

import numpy as np
import torch

from . import _io
from . import distributed as D
from .autoencoder import get_autoencoder
from .ddpm import RULES, cached_sampler, ddim_timesteps
from .uvit import UViT


class _Rule:
    """Stand-in for the reference's post-processing callables (sampler.py:47-79): identifies the update rule the
    fused DDPM kernel applies; it is not called per step."""

    def __init__(self, name: str):
        self.name = name

    def __repr__(self):
        return f"<{self.name}_postprocessing>"


predict_noise_postprocessing = _Rule("predict_noise")
predict_original_postprocessing = _Rule("predict_original")
predict_previous_postprocessing = _Rule("predict_previous")
_BY_NAME = {r.name: r for r in (predict_noise_postprocessing, predict_original_postprocessing,
                                predict_previous_postprocessing)}


def _rule_name(postprocessing) -> str:
    if isinstance(postprocessing, _Rule):
        return postprocessing.name
    if isinstance(postprocessing, str) and postprocessing in RULES:
        return postprocessing
    name = getattr(postprocessing, "__name__", "")
    for r in RULES:  # the reference's own function objects are accepted by name
        if name == f"{r}_postprocessing":
            return r
    raise ValueError(f"unsupported postprocessing {postprocessing!r}; expected one of {RULES}")


def _pick_device(model, device=None) -> torch.device:
    """The reference samples on its module-level `device` (sampler.py:37); here: the explicit argument, else the device
    the model's parameters live on, else the current CUDA device."""
    if device is not None:
        return torch.device(device)
    mdev = getattr(model, "device", None)
    if isinstance(mdev, torch.device) and mdev.type == "cuda":
        return mdev
    return torch.device("cuda", torch.cuda.current_device())


def _ddim_plan(ddim_steps: int, late_available: bool, t_switch):
    """(timesteps, late flags) of the DDIM loop, sampler.py:103-123: pairs (t, s) of the strided schedule; the
    hand-off `if t < 1000 - t_switch: model = late_model` happens AFTER the step at t."""
    ts = ddim_timesteps(ddim_steps)
    steps, flags, on_late = ts[:-1], [], False
    for t in steps:
        flags.append(on_late)
        if late_available and t < 1000 - t_switch:
            on_late = True
    return steps, flags


def get_samples(model, batch_size: int, postprocessing, seed: int, num_channels: int, sample_height: int,
                sample_width: int, use_ddim: bool = False, ddim_steps: int = 50, ddim_eta: float = 0.0,
                timesteps_save: List[int] = (), y=None, autoencoder=None, late_model=None, t_switch=np.inf, *,
                noise=None, use_graph: bool = True, device=None, x_T=None, noise_row_offset: int = 0):
    """sampler.py:82-155.  Returns (samples [B,H,W,C] f32 numpy un-clipped, [intermediate samples]).

    x_T is drawn on the CPU generator after ``seed_everything(seed)`` exactly like the reference (sampler.py:99-100);
    the per-step z comes from an in-kernel Philox stream keyed by ``seed`` unless ``noise`` [1000,B,C,H,W] (indexed
    by t) is injected (parity tests).  ``use_ddim`` runs the strided DDIM branch (sampler.py:103-126, including the
    reference's sigma_t^2 * z noise term).  ``autoencoder`` (duodiff_b200.autoencoder.get_autoencoder, or any object
    with the reference's ``decode``) maps the final and the saved intermediate latents to images (sampler.py:141-143,
    149-150).

    Sharded (data-parallel) use, see duodiff_b200.distributed: ``x_T`` [B,C,H,W] replaces the draw of the initial
    noise (this rank's rows of the global draw) and ``noise_row_offset`` is the global index of its first row, which
    keys the Philox stream -- the shards of a global batch then reproduce the single-process result row for row."""
    dev = _pick_device(model, device)
    _io.seed_everything(seed)
    if x_T is None:
        x = torch.randn(batch_size, num_channels, sample_height, sample_width)
    else:
        x = torch.as_tensor(x_T, dtype=torch.float32).detach().cpu().contiguous()
        if tuple(x.shape) != (batch_size, num_channels, sample_height, sample_width):
            raise ValueError(f"x_T has shape {tuple(x.shape)}, expected "
                             f"{(batch_size, num_channels, sample_height, sample_width)}")
    x = x.pin_memory().to(dev, non_blocking=True)
    with torch.cuda.device(dev):
        early = model.engine(batch_size)
        late = late_model.engine(batch_size) if late_model is not None else None
        if noise is not None:
            noise = noise.to(device=dev, dtype=torch.float32).contiguous()
        # reference: `if 1000 - t in timesteps_save` after the update at t -> save x after the step at t = 1000 - s
        save_at = {1000 - int(s) for s in timesteps_save}
        kept = []

        def finalize(lat):
            if autoencoder:
                print("Decode the images...")
                lat = autoencoder.decode(lat).contiguous()
            return sampler.finalize(lat)
        if use_ddim:
            sampler = cached_sampler(early, late, t_switch, batch_size, rule=("ddim", int(ddim_steps), float(ddim_eta)))
            sampler.set_noise_offset(noise_row_offset)
            steps, flags = _ddim_plan(int(ddim_steps), late is not None, t_switch)
            k0 = 0
            for k, t in enumerate(steps):
                if t in save_at or k == len(steps) - 1:
                    sampler.run_list(x, steps[k0:k + 1], flags[k0:k + 1], y=y, noise=noise, seed=seed,
                                     use_graph=use_graph)
                    if t in save_at:
                        kept.append(finalize(x))
                    k0 = k + 1
        else:
            sampler = cached_sampler(early, late, t_switch, batch_size, rule=_rule_name(postprocessing))
            sampler.set_noise_offset(noise_row_offset)
            t_first = 999
            for t_stop in sorted((t for t in save_at if 0 <= t <= 999), reverse=True) + [0]:
                if t_stop > t_first:
                    continue
                sampler.run(x, y=y, noise=noise, seed=seed, t_first=t_first, t_last=t_stop, use_graph=use_graph)
                if t_stop in save_at:
                    kept.append(finalize(x))
                t_first = t_stop - 1
                if t_first < 0:
                    break
        samples = finalize(x)
        out = samples.cpu().numpy()
        # the reference appends in loop order (descending t), one entry per matching step
        inter = [k.cpu().numpy() for k in kept]
    return out, inter


def dump_samples(samples, output_folder: Path, timestep=1000):
    _io.dump_samples(samples, output_folder, timestep)


def dump_statistics(elapsed_time, output_folder: Path):
    """sampler.py:187-189."""
    with open(Path(output_folder) / "statistics.txt", "w") as f:
        f.write(f"Elapsed time: {elapsed_time} s\n")


def get_args(argv=None):
    p = ArgumentParser()
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--checkpoint_path", type=str, required=True, help="Path to checkpoint of the model")
    p.add_argument("--checkpoint_path_late", type=str, default=None,
                   help="Path to checkpoint of the model to be used in the latest steps")
    p.add_argument("--batch_size", type=int, required=True)
    p.add_argument("--parametrization", type=str, choices=list(RULES), required=True)
    p.add_argument("--output_folder", type=str, required=True)
    p.add_argument("--config_path", type=str, required=True, help="Path to yaml config file")
    p.add_argument("--config_path_late", type=str, default=None,
                   help="Path to yaml config file of the model to be used in the latest steps")
    p.add_argument("--t_switch", type=int, default=np.inf,
                   help="Sampling timestep where the model should be replaced by the late model")
    p.add_argument("--class_id", type=int, default=None, help="Number up to 1000 that corresponds to a class")
    p.add_argument("--use_ddim", action="store_true")
    p.add_argument("--ddim_steps", type=int, default=50)
    p.add_argument("--ddim_eta", type=float, default=0.0)
    p.add_argument("--timesteps_save", type=int, nargs="+", default=[])
    return p.parse_args(argv)


def draw_labels(batch_size: int, num_classes: int):
    """sampler.py:314-318 / eesampler.py:176-180: with --class_id the reference draws a RANDOM label per sample,
    ``torch.randint(1, 1001, (batch_size,))`` (Q14; the flag's value is ignored).  Deviation, stated: that range
    overflows a 1000-row embedding table (label 1000 -> IndexError in the reference, 1 time in 1000 per sample), so the
    labels are taken modulo ``num_classes`` here; for every label the reference can embed the value is unchanged."""
    y = torch.randint(1, 1001, (batch_size,))
    return y % num_classes if num_classes > 0 else y


def _build(config_path, checkpoint_path, batch_size, device):
    cfg = _io.load_config(config_path)
    net = UViT(**_io.uvit_kwargs(cfg), max_batch=batch_size)
    _io.load_checkpoint_into(net, checkpoint_path)
    return net.eval().to(device), cfg


def main(argv=None):
    """The reference's CLI.  Under `torchrun --nproc-per-node N` each rank samples its shard of the --batch_size
    images (duodiff_b200.distributed) and rank 0 writes exactly the files a single process writes."""
    args = get_args(argv)
    out_dir = Path(args.output_folder)
    if D.env_rank_world()[0] == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
    if not torch.cuda.is_available():
        raise RuntimeError("duodiff_b200.sampler needs a B200 (sm_100) GPU; there is no CPU path")
    with D.cli_process_group() as (rank, world, device):
        print(f"Using device {device}")
        lo, hi = D.shard_bounds(args.batch_size, rank, world)
        model = late = autoencoder = None
        if hi > lo:  # a rank with an empty shard (more ranks than images) builds nothing
            model, cfg = _build(args.config_path, args.checkpoint_path, hi - lo, device)
            if args.checkpoint_path_late:
                late, cfg = _build(args.config_path_late, args.checkpoint_path_late, hi - lo, device)
        else:
            cfg = _io.load_config(args.config_path_late if args.checkpoint_path_late else args.config_path)
        mp = cfg["model_params"]
        _io.seed_everything(args.seed)
        y = None
        if args.class_id is not None:
            y = draw_labels(args.batch_size, mp.get("num_classes", -1)).to(device)
        if "autoencoder" in cfg and hi > lo:  # sampler.py:320-325
            autoencoder = get_autoencoder(cfg["autoencoder"]["autoencoder_checkpoint_path"])
        D.barrier()  # every rank has loaded its models: the clock starts together
        tic = time.time()
        local = D.run_shard(
            functools.partial(get_samples, model=model), args.batch_size,
            shape=(mp["in_chans"], mp["img_size"], mp["img_size"]), seed=args.seed, y=y,
            postprocessing=_BY_NAME[args.parametrization], num_channels=mp["in_chans"],
            sample_height=mp["img_size"], sample_width=mp["img_size"], use_ddim=args.use_ddim,
            ddim_steps=args.ddim_steps, ddim_eta=args.ddim_eta, autoencoder=autoencoder, late_model=late,
            t_switch=args.t_switch, timesteps_save=args.timesteps_save)
        D.barrier()  # every shard is done: what follows is the gather alone
        t_gather = time.time()
        result = D.gather_to_rank0(local, args.batch_size, D.SAMPLER_OUTPUTS)
        tac = time.time()
        if rank != 0:
            return
        if world > 1:
            print(f"Gathered {args.batch_size} samples from {world} ranks in {tac - t_gather:.3f} s")
        samples, inter = result
        dump_statistics(tac - tic, out_dir)
        dump_samples(samples, out_dir)
        if args.timesteps_save:
            for ts, s in zip(args.timesteps_save, inter):
                dump_samples(s, out_dir, ts)


if __name__ == "__main__":
    main()
