"""Drop-in for the reference's ``sampler.py``: same ``get_samples`` signature and CLI flags (sampler.py:82-155,192-252),
but the 1000-step loop — U-ViT forwards, the DuoDiff hand-off after ``t == 1000 - t_switch`` and the per-step DDPM
update — runs inside libduodiff_b200.so as CUDA-graph replays of hand-written sm_100a kernels.

    python -m duodiff_b200.sampler --checkpoint_path early.pth --config_path configs/uvit_celeba_3.yaml \
        --checkpoint_path_late full.pth --config_path_late configs/uvit_celeba.yaml --t_switch 300 \
        --batch_size 128 --parametrization predict_noise --output_folder out/
"""
from __future__ import annotations

import functools
import math
import time
from argparse import SUPPRESS, ArgumentParser
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


def _guidance(models, y, cfg_scale, null_label):
    """(scale, null_label) of classifier-free guidance, checked against every backbone of the run."""
    from .early_exit import EarlyExitUViT
    if y is None:
        raise ValueError("cfg_scale needs class labels y: guidance contrasts y with the null label")
    for m in models:
        if isinstance(m, EarlyExitUViT):
            raise ValueError("cfg_scale is not supported with early exit: the conditional and unconditional rows "
                             "would leave at different layers")
        if getattr(m, "num_classes", 0) <= 0:
            raise ValueError("cfg_scale needs a class-conditional model (num_classes > 0)")
    scale = float(cfg_scale)
    if not math.isfinite(scale):
        raise ValueError(f"cfg_scale must be finite, got {cfg_scale!r}")
    # U-ViT's convention: the last row of the label table is the null ("unconditional") label
    null = models[0].num_classes - 1 if null_label is None else int(null_label)
    for m in models:
        if not 0 <= null < m.num_classes:
            raise ValueError(f"null_label {null} is outside [0, {m.num_classes})")
    return scale, null


def _dpm_solver_rule(models, postprocessing, use_ddim, steps):
    """Sampler rule ("dpm_solver++", steps, parametrization) of DPM-Solver++(2M), checked against the run."""
    from .early_exit import EarlyExitUViT
    if use_ddim:
        raise ValueError("dpm_solver_steps and use_ddim select two different samplers: give one of them")
    name = _rule_name(postprocessing)
    if name == "predict_previous":
        raise ValueError("DPM-Solver++ needs a noise or data prediction, not predict_previous")
    if int(steps) < 2:
        raise ValueError(f"dpm_solver_steps={steps}: the grid needs at least 2 points (one model evaluation)")
    if any(isinstance(m, EarlyExitUViT) for m in models):
        raise ValueError("dpm_solver_steps is not supported with early exit")
    return "dpm_solver++", int(steps), name


def _unipc_rule(models, postprocessing, use_ddim, dpm_solver_steps, steps):
    """Sampler rule ("unipc", steps, parametrization) of UniPC, checked against the run."""
    from .early_exit import EarlyExitUViT
    if use_ddim or dpm_solver_steps is not None:
        raise ValueError("unipc_steps, use_ddim and dpm_solver_steps select different samplers: give one of them")
    name = _rule_name(postprocessing)
    if name == "predict_previous":
        raise ValueError("UniPC needs a noise or data prediction, not predict_previous")
    if int(steps) < 2:
        raise ValueError(f"unipc_steps={steps}: the grid needs at least 2 points (one model evaluation)")
    if any(isinstance(m, EarlyExitUViT) for m in models):
        raise ValueError("unipc_steps is not supported with early exit")
    return "unipc", int(steps), name


def _sde_dpm_solver_rule(models, postprocessing, use_ddim, dpm_solver_steps, unipc_steps, steps):
    """Sampler rule ("sde-dpm_solver++", steps, parametrization) of SDE-DPM-Solver++(2M), checked against the run."""
    from .early_exit import EarlyExitUViT
    if use_ddim or dpm_solver_steps is not None or unipc_steps is not None:
        raise ValueError("sde_dpm_solver_steps, use_ddim, dpm_solver_steps and unipc_steps select different samplers: "
                         "give one of them")
    name = _rule_name(postprocessing)
    if name == "predict_previous":
        raise ValueError("SDE-DPM-Solver++ needs a noise or data prediction, not predict_previous")
    if int(steps) < 2:
        raise ValueError(f"sde_dpm_solver_steps={steps}: the grid needs at least 2 points (one model evaluation)")
    if any(isinstance(m, EarlyExitUViT) for m in models):
        raise ValueError("sde_dpm_solver_steps is not supported with early exit")
    return "sde-dpm_solver++", int(steps), name


def get_samples(model, batch_size: int, postprocessing, seed: int, num_channels: int, sample_height: int,
                sample_width: int, use_ddim: bool = False, ddim_steps: int = 50, ddim_eta: float = 0.0,
                timesteps_save: List[int] = (), y=None, autoencoder=None, late_model=None, t_switch=np.inf, *,
                noise=None, use_graph: bool = True, device=None, x_T=None, noise_row_offset: int = 0,
                cfg_scale=None, null_label=None, dpm_solver_steps=None, unipc_steps=None, sde_dpm_solver_steps=None):
    """sampler.py:82-155.  Returns (samples [B,H,W,C] f32 numpy un-clipped, [intermediate samples]).

    x_T is drawn on the CPU generator after ``seed_everything(seed)`` exactly like the reference (sampler.py:99-100);
    the per-step z comes from an in-kernel Philox stream keyed by ``seed`` unless ``noise`` [1000,B,C,H,W] (indexed
    by t) is injected (parity tests).  ``use_ddim`` runs the strided DDIM branch (sampler.py:103-126, including the
    reference's sigma_t^2 * z noise term).  ``autoencoder`` (duodiff_b200.autoencoder.get_autoencoder, or any object
    with the reference's ``decode``) maps the final and the saved intermediate latents to images (sampler.py:141-143,
    149-150).

    Sharded (data-parallel) use, see duodiff_b200.distributed: ``x_T`` [B,C,H,W] replaces the draw of the initial
    noise (this rank's rows of the global draw) and ``noise_row_offset`` is the global index of its first row, which
    keys the Philox stream -- the shards of a global batch then reproduce the single-process result row for row.

    Classifier-free guidance (not in the reference): with ``cfg_scale`` s every step runs the backbone on 2B rows,
    labels ``y`` and ``null_label`` (default num_classes - 1, U-ViT's null row), and uses eps = eps_c + s * (eps_c -
    eps_u); s = 0 gives the unguided samples.  It helps only checkpoints trained with label dropout to that row.
    ``cfg_scale=None`` runs the unguided path unchanged.

    DPM-Solver++(2M) (not in the reference): ``dpm_solver_steps`` n runs the second-order multistep solver of the
    probability-flow ODE over the DDIM grid (n - 1 model evaluations at the timesteps of ``use_ddim=True,
    ddim_steps=n``), with the hand-off, ``timesteps_save``, ``autoencoder`` and ``cfg_scale`` as in the DDIM branch.
    It has no noise term.  ``postprocessing`` must be predict_noise or predict_original.

    UniPC (not in the reference): ``unipc_steps`` n runs the second-order predictor-corrector solver of the same ODE
    (bh2, data prediction) over the same grid and with the same options as ``dpm_solver_steps``.  The corrector reuses
    each step's model evaluation, so n - 1 evaluations still suffice; the final step is first order.  A saved
    intermediate is the predicted x the next evaluation sees (its correction needs that evaluation).

    SDE-DPM-Solver++(2M) (not in the reference): ``sde_dpm_solver_steps`` n runs the second-order multistep solver of
    the reverse SDE over the same grid and with the same options as ``dpm_solver_steps``.  Each step but the final one
    adds noise, the draw the DDPM step at that t makes (``seed`` or ``noise[t]``); a first-order step is the DDPM
    posterior step between the two grid points.  The first and the final step are first order.  A saved intermediate
    is x after that step, its noise included."""
    models = [m for m in (model, late_model) if m is not None]
    guidance = None
    if cfg_scale is not None:
        guidance = _guidance(models, y, cfg_scale, null_label)
    solver_rule = None  # DPM-Solver++, UniPC or SDE-DPM-Solver++
    if dpm_solver_steps is not None:
        solver_rule = _dpm_solver_rule(models, postprocessing, use_ddim, dpm_solver_steps)
    if unipc_steps is not None:
        solver_rule = _unipc_rule(models, postprocessing, use_ddim, dpm_solver_steps, unipc_steps)
    if sde_dpm_solver_steps is not None:
        solver_rule = _sde_dpm_solver_rule(models, postprocessing, use_ddim, dpm_solver_steps, unipc_steps,
                                           sde_dpm_solver_steps)
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
        rows = batch_size if guidance is None else 2 * batch_size  # guided forwards run on [x ; x]
        early = model.engine(rows)
        late = late_model.engine(rows) if late_model is not None else None
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
        if use_ddim or solver_rule is not None:
            # DDIM and the DPM-Solver++ / UniPC / SDE solvers walk the same grid; after the step at t in save_at x is
            # saved
            rule = solver_rule or ("ddim", int(ddim_steps), float(ddim_eta))
            sampler = cached_sampler(early, late, t_switch, batch_size, rule=rule, guidance=guidance)
            sampler.set_noise_offset(noise_row_offset)
            steps, flags = _ddim_plan(rule[1], late is not None, t_switch)
            k0 = 0
            for k, t in enumerate(steps):
                if t in save_at or k == len(steps) - 1:
                    sampler.run_list(x, steps[k0:k + 1], flags[k0:k + 1], y=y, noise=noise, seed=seed,
                                     use_graph=use_graph)
                    if t in save_at:
                        kept.append(finalize(x))
                    k0 = k + 1
        else:
            sampler = cached_sampler(early, late, t_switch, batch_size, rule=_rule_name(postprocessing),
                                     guidance=guidance)
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
    # not a flag of the reference: absent from the namespace unless given, so unguided runs parse exactly as before
    p.add_argument("--cfg_scale", type=float, default=SUPPRESS,
                   help="Classifier-free guidance scale s: eps = eps_c + s * (eps_c - eps_u) against the null label "
                        "num_classes - 1 (needs --class_id)")
    p.add_argument("--dpm_solver_steps", type=int, default=SUPPRESS,
                   help="Sample with DPM-Solver++(2M) over the DDIM grid of N points (N - 1 model evaluations, the "
                        "timesteps of --use_ddim --ddim_steps N); no noise term")
    p.add_argument("--unipc_steps", type=int, default=SUPPRESS,
                   help="Sample with UniPC (bh2, second-order predictor-corrector) over the DDIM grid of N points (N - 1 "
                        "model evaluations, the timesteps of --use_ddim --ddim_steps N); no noise term")
    p.add_argument("--sde_dpm_solver_steps", type=int, default=SUPPRESS,
                   help="Sample with SDE-DPM-Solver++(2M), the stochastic second-order multistep solver, over the DDIM "
                        "grid of N points (N - 1 model evaluations, the timesteps of --use_ddim --ddim_steps N); every "
                        "step but the final one adds noise")
    args = p.parse_args(argv)
    if getattr(args, "cfg_scale", None) is not None and args.class_id is None:
        p.error("--cfg_scale needs --class_id: guidance contrasts the class labels with the null label")
    if getattr(args, "dpm_solver_steps", None) is not None:
        if args.use_ddim:
            p.error("--dpm_solver_steps and --use_ddim select two different samplers: give one of them")
        if args.parametrization == "predict_previous":
            p.error("--dpm_solver_steps needs --parametrization predict_noise or predict_original")
        if args.dpm_solver_steps < 2:
            p.error("--dpm_solver_steps needs at least 2 grid points (one model evaluation)")
    if getattr(args, "unipc_steps", None) is not None:
        if args.use_ddim or getattr(args, "dpm_solver_steps", None) is not None:
            p.error("--unipc_steps, --use_ddim and --dpm_solver_steps select different samplers: give one of them")
        if args.parametrization == "predict_previous":
            p.error("--unipc_steps needs --parametrization predict_noise or predict_original")
        if args.unipc_steps < 2:
            p.error("--unipc_steps needs at least 2 grid points (one model evaluation)")
    if getattr(args, "sde_dpm_solver_steps", None) is not None:
        if args.use_ddim or getattr(args, "dpm_solver_steps", None) is not None or \
                getattr(args, "unipc_steps", None) is not None:
            p.error("--sde_dpm_solver_steps, --use_ddim, --dpm_solver_steps and --unipc_steps select different "
                    "samplers: give one of them")
        if args.parametrization == "predict_previous":
            p.error("--sde_dpm_solver_steps needs --parametrization predict_noise or predict_original")
        if args.sde_dpm_solver_steps < 2:
            p.error("--sde_dpm_solver_steps needs at least 2 grid points (one model evaluation)")
    return args


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
    cfg_scale = getattr(args, "cfg_scale", None)
    out_dir = Path(args.output_folder)
    if D.env_rank_world()[0] == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
    if not torch.cuda.is_available():
        raise RuntimeError("duodiff_b200.sampler needs a B200 (sm_100) GPU; there is no CPU path")
    with D.cli_process_group() as (rank, world, device):
        print(f"Using device {device}")
        lo, hi = D.shard_bounds(args.batch_size, rank, world)
        model = late = autoencoder = None
        rows = (hi - lo) * (2 if cfg_scale is not None else 1)  # a guided forward runs on 2B rows
        if hi > lo:  # a rank with an empty shard (more ranks than images) builds nothing
            model, cfg = _build(args.config_path, args.checkpoint_path, rows, device)
            if args.checkpoint_path_late:
                late, cfg = _build(args.config_path_late, args.checkpoint_path_late, rows, device)
        else:
            cfg = _io.load_config(args.config_path_late if args.checkpoint_path_late else args.config_path)
        mp = cfg["model_params"]
        _io.seed_everything(args.seed)
        y = None
        if args.class_id is not None:
            y = draw_labels(args.batch_size, mp.get("num_classes", -1)).to(device)
        extra = {}  # keywords of the samplers that are not in the reference
        if cfg_scale is not None:
            extra = dict(cfg_scale=cfg_scale, null_label=mp.get("num_classes", -1) - 1)
            if rank == 0:
                print(f"Classifier-free guidance: scale {cfg_scale}, null label {extra['null_label']} "
                      f"(the last row of the {mp.get('num_classes', -1)}-row label table)")
        if getattr(args, "dpm_solver_steps", None) is not None:
            extra["dpm_solver_steps"] = args.dpm_solver_steps
        if getattr(args, "unipc_steps", None) is not None:
            extra["unipc_steps"] = args.unipc_steps
        if getattr(args, "sde_dpm_solver_steps", None) is not None:
            extra["sde_dpm_solver_steps"] = args.sde_dpm_solver_steps
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
            t_switch=args.t_switch, timesteps_save=args.timesteps_save, **extra)
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
