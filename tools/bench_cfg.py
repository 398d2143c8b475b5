"""Classifier-free guidance on the ImageNet-256 DuoDiff pair (imagenet256_3 -> imagenet256, t_switch 300, random-init
weights, 1001 classes):

  * in-graph step time (CUDA events around replays of the captured step graphs, per backbone) of guided sampling at
    B = 128 next to unguided sampling at B = 256: both run the backbones on 256 rows, so the difference is the cost
    of the guided tail (two bands staged and convolved, two heads written);
  * guided images/s at B = 128 through get_samples(cfg_scale=...): 1000-step DDPM and 50-step DDIM, without and with
    the KL-f8 decode to 256x256 (random-init autoencoder); unguided DDIM at B = 256 for comparison;
  * the card's name and power limit, read in the same run.

    python tools/bench_cfg.py --out profiles/r04_cfg.txt
"""
from __future__ import annotations

import argparse
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"not read ({e})"


def step_ms(smp, x, y, t_first, t_last, reps=3):
    """Mean in-graph time of one step over the window t_first..t_last (graphs captured by a warm-up run)."""
    smp.run(x.clone(), y=y, seed=1, t_first=t_first, t_last=t_last)
    best = []
    for _ in range(reps):
        xs = x.clone()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        smp.run(xs, y=y, seed=1, t_first=t_first, t_last=t_last)
        b.record()
        torch.cuda.synchronize()
        best.append(a.elapsed_time(b) / (t_first - t_last + 1))
    return min(best), max(best)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", type=Path, required=True)
    ap.add_argument("--batch", type=int, default=128)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cfg needs a B200: there is no CPU measurement")
    import duodiff_b200 as ddb
    from duodiff_b200 import sampler as S
    from duodiff_b200.autoencoder import get_autoencoder
    from duodiff_b200.configs import CONFIGS
    from duodiff_b200.ddpm import Sampler
    from oracle.ae_oracle import AESpec, random_state_dict

    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card (name, power.limit, clocks.max.sm): {card()}")
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    early = ddb.UViT(**CONFIGS["imagenet256_3"], max_batch=2 * args.batch).eval().to(dev)
    late = ddb.UViT(**CONFIGS["imagenet256"], max_batch=2 * args.batch).eval().to(dev)
    B, B2 = args.batch, 2 * args.batch
    log(f"ImageNet-256 DuoDiff pair, t_switch 300, random-init weights, 1001 classes; guided B = {B}, "
        f"unguided B = {B2} (both {B2} forward rows); cfg_scale 1.5, null label 1000")
    e, l_ = early.engine(B2), late.engine(B2)
    g = torch.Generator(device=dev).manual_seed(1)
    y2 = torch.randint(0, 1000, (B2,), device=dev, generator=g)
    x2 = torch.randn(B2, 4, 32, 32, device=dev, generator=g)
    guided = Sampler(e, l_, 300, B, guidance=(1.5, 1000))
    plain = Sampler(e, l_, 300, B2)
    for name, (t0, t1) in (("early (imagenet256_3)", (999, 900)), ("late (imagenet256)", (599, 500))):
        # alternate the two so that clock drift hits both alike
        pg, pp = [], []
        for _ in range(2):
            pg.append(step_ms(guided, x2[:B].contiguous(), y2[:B].contiguous(), t0, t1))
            pp.append(step_ms(plain, x2, y2, t0, t1))
        g_ms, p_ms = min(v[0] for v in pg), min(v[0] for v in pp)
        spread = max(v[1] for v in pg + pp) / min(v[0] for v in pg + pp) - 1
        log(f"step on the {name} backbone, t = {t0}..{t1}: guided B = {B} {g_ms:.3f} ms, unguided B = {B2} "
            f"{p_ms:.3f} ms, difference {1e3 * (g_ms - p_ms):+.1f} us ({100 * (g_ms / p_ms - 1):+.2f} %); "
            f"spread of all windows {100 * spread:.1f} %")
    for k in ("tail",):
        pg = guided.profile_step(x2[:B].clone(), 999, False, y=y2[:B].contiguous())[k]
        pp = plain.profile_step(x2.clone(), 999, False, y=y2)[k]
        log(f"eager step, event-timed '{k}' kernel: guided B = {B} {1e3 * pg['ms']:.1f} us, unguided B = {B2} "
            f"{1e3 * pp['ms']:.1f} us (profiling timestamps every kernel: slower than the graph)")
    del guided, plain

    with tempfile.TemporaryDirectory() as tmp:
        ae_path = Path(tmp) / "ae.pth"
        torch.save(random_state_dict(AESpec(), 3), ae_path)
        ae = get_autoencoder(str(ae_path))
        yc = y2[:B].cpu()
        kw = dict(postprocessing=S.predict_noise_postprocessing, seed=0, num_channels=4, sample_height=32,
                  sample_width=32, late_model=late, t_switch=300)

        def rate(label, batch, **extra):
            S.get_samples(early, batch, **kw, **dict(extra, use_ddim=True, ddim_steps=5))  # warm-up: engines, graphs
            torch.cuda.synchronize()
            tic = time.perf_counter()
            out, _ = S.get_samples(early, batch, **kw, **extra)
            torch.cuda.synchronize()
            dt = time.perf_counter() - tic
            log(f"{label}: {batch} images in {dt:.3f} s -> {batch / dt:.2f} images/s (finite: "
                f"{bool(np.isfinite(out).all())})")
            return batch / dt

        rate(f"guided DDIM 50 steps, B = {B}, no decode", B, y=yc, cfg_scale=1.5, use_ddim=True, ddim_steps=50)
        rate(f"unguided DDIM 50 steps, B = {B2}, no decode", B2, y=y2.cpu(), use_ddim=True, ddim_steps=50)
        rate(f"guided DDIM 50 steps, B = {B}, with decode", B, y=yc, cfg_scale=1.5, use_ddim=True, ddim_steps=50,
             autoencoder=ae)
        rate(f"guided DDPM 1000 steps, B = {B}, no decode", B, y=yc, cfg_scale=1.5)
        rate(f"guided DDPM 1000 steps, B = {B}, with decode", B, y=yc, cfg_scale=1.5, autoencoder=ae)
    log("unguided DDPM 1000 steps at B = 256: not measured")
    log(f"card after the runs: {card()}")
    args.out.parent.mkdir(parents=True, exist_ok=True)
    args.out.write_text("# python tools/bench_cfg.py (one B200)\n" + "\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
