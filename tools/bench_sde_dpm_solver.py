"""SDE-DPM-Solver++(2M) against DPM-Solver++(2M) and DDIM on the DuoDiff pairs (t_switch 300, random-init weights):

  * in-graph step time (CUDA events around whole replayed trajectories over the same 50-point grid, so the three
    samplers run the same timesteps on the same backbones, alternated) of DDIM (eta 0), DPM-Solver++ and
    SDE-DPM-Solver++: guided ImageNet-256 (imagenet256_3 -> imagenet256, cfg_scale 1.5) at B = 128 and CelebA
    (celeba_3 -> celeba) at B = 128.  The SDE tail does the DPM-Solver++ tail's work plus the Philox draw of the DDPM
    tail;
  * the eager, event-timed tail kernel on an order-2 row (t = 958 of the 50-point grid) and on the first row;
  * guided ImageNet-256 images/s at B = 128 with the KL-f8 decode (random-init autoencoder) through get_samples:
    DPM-Solver++ and SDE-DPM-Solver++ at n in {11, 16, 21, 26}, alternated;
  * the card's name and power limit, read in the same run.
No FID is computed (the Inception weights are not available).

    python tools/bench_sde_dpm_solver.py --out profiles/r08_sde_dpm_solver.txt
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


def traj_ms(smp, x, y, steps, flags, reps=3):
    """(min, max) in-graph time per step of whole replayed trajectories (graphs captured by a warm-up run)."""
    smp.run_list(x.clone(), steps, flags, y=y, seed=1)
    out = []
    for _ in range(reps):
        xs = x.clone()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        smp.run_list(xs, steps, flags, y=y, seed=1)
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / len(steps))
    return min(out), max(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", type=Path, required=True)
    ap.add_argument("--batch", type=int, default=128)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sde_dpm_solver needs a B200: there is no CPU measurement")
    import duodiff_b200 as ddb
    from duodiff_b200 import sampler as S
    from duodiff_b200.autoencoder import get_autoencoder
    from duodiff_b200.configs import CONFIGS
    from duodiff_b200.ddpm import Sampler
    from duodiff_b200.sampler import _ddim_plan
    from oracle.ae_oracle import AESpec, random_state_dict

    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card (name, power.limit, clocks.max.sm): {card()}")
    dev = torch.device("cuda:0")
    B = args.batch
    steps, flags = _ddim_plan(50, True, 300)
    names = ("DDIM", "DPM-Solver++", "SDE-DPM-Solver++")
    for pair, guided in ((("imagenet256_3", "imagenet256"), True), (("celeba_3", "celeba"), False)):
        torch.manual_seed(0)
        rows = 2 * B if guided else B
        early = ddb.UViT(**CONFIGS[pair[0]], max_batch=rows).eval().to(dev)
        late = ddb.UViT(**CONFIGS[pair[1]], max_batch=rows).eval().to(dev)
        C, H = early.in_chans, early.img_size
        g = torch.Generator(device=dev).manual_seed(1)
        x = torch.randn(B, C, H, H, device=dev, generator=g)
        y = torch.randint(0, 1000, (B,), device=dev, generator=g) if guided else None
        gd = (1.5, early.num_classes - 1) if guided else None
        e, l_ = early.engine(rows), late.engine(rows)
        smps = [Sampler(e, l_, 300, B, rule=r, guidance=gd)
                for r in (("ddim", 50, 0.0), ("dpm_solver++", 50, "predict_noise"),
                          ("sde-dpm_solver++", 50, "predict_noise"))]
        runs = [[] for _ in smps]
        for _ in range(3):  # alternate the three so that clock drift hits all alike
            for i, smp in enumerate(smps):
                runs[i].append(traj_ms(smp, x, y, steps, flags))
        best = [min(v[0] for v in r) for r in runs]
        spread = max(v[1] for r in runs for v in r) / min(v[0] for r in runs for v in r) - 1
        log(f"{pair[0]} -> {pair[1]}{' guided' if guided else ''}, B = {B}, 50-point grid (49 steps, "
            f"{sum(flags)} on the late backbone): " + ", ".join(f"{n} {ms:.3f} ms/step" for n, ms in zip(names, best))
            + f"; SDE - DDIM {1e3 * (best[2] - best[0]):+.1f} us ({100 * (best[2] / best[0] - 1):+.2f} %), "
            f"SDE - DPM-Solver++ {1e3 * (best[2] - best[1]):+.1f} us ({100 * (best[2] / best[1] - 1):+.2f} %); "
            f"spread of all runs {100 * spread:.1f} %")
        # t = 958: an order-2 row of the 50-point grid (D_prev read, Philox drawn); profile_step draws Philox noise
        for t in (999, 958):
            v = [min(smp.profile_step(x.clone(), t, False, y=y)["tail"]["ms"] for _ in range(3)) for smp in smps]
            log(f"  eager step at t = {t}, event-timed 'tail' kernel (best of 3): " +
                ", ".join(f"{n} {1e3 * ms:.1f} us" for n, ms in zip(names, v)) +
                " (profiling timestamps every kernel: slower than the graph)")
        del smps
        if not guided:
            del early, late
            continue

        with tempfile.TemporaryDirectory() as tmp:
            ae_path = Path(tmp) / "ae.pth"
            torch.save(random_state_dict(AESpec(), 3), ae_path)
            ae = get_autoencoder(str(ae_path))
            kw = dict(postprocessing=S.predict_noise_postprocessing, seed=0, num_channels=4, sample_height=32,
                      sample_width=32, late_model=late, t_switch=300, y=y.cpu(), cfg_scale=1.5, autoencoder=ae)

            def rate(label, **extra):
                S.get_samples(early, B, **kw, **extra)  # warm-up: engines, graphs, decoder
                torch.cuda.synchronize()
                tic = time.perf_counter()
                out, _ = S.get_samples(early, B, **kw, **extra)
                torch.cuda.synchronize()
                dt = time.perf_counter() - tic
                log(f"{label}: {B} images in {dt:.3f} s -> {B / dt:.2f} images/s (finite: "
                    f"{bool(np.isfinite(out).all())})")

            for n in (11, 16, 21, 26):
                rate(f"guided DPM-Solver++ {n} points ({n - 1} evaluations), with decode", dpm_solver_steps=n)
                rate(f"guided SDE-DPM-Solver++ {n} points ({n - 1} evaluations), with decode",
                     sde_dpm_solver_steps=n)
        del early, late
    log("FID: not measured (the Inception weights are not available)")
    log(f"card after the runs: {card()}")
    args.out.parent.mkdir(parents=True, exist_ok=True)
    args.out.write_text("# python tools/bench_sde_dpm_solver.py (one B200)\n" + "\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
