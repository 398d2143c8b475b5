"""DDIM sampling with early exit on BASELINE config 3 (bench.py --ee: CelebA deediff, mlp_probe_per_layer, threshold
0.08, B = 128, compaction mode; random-init backbone with bench.synthetic_probes_, slope 1.0 / wscale 0.5):

  * images/s through eesampler.get_samples (x_T draw, sampling, epilogue, copy to the host) for 1000-step DDPM,
    DDIM 100 and DDIM 50 (eta 0), at threshold 0.08 and at threshold 0.0 (no sample ever exits);
  * the mean exit layer over the visited timesteps and the in-graph step time (CUDA events around replayed whole
    trajectories) of each;
  * whether the probes, calibrated over the 1000-step trajectory, exit at the same layers on the DDIM grid: the DDPM
    run's mean exit layer at the grid's timesteps against the DDIM run's, per timestep band.  Random-init weights:
    this says how the synthetic probes react to the coarser trajectory, not what a trained probe does;
  * the card's name and power limit, read in the same run.  FID: not measured (the Inception weights are not
    available).

    python tools/bench_ee_ddim.py --out profiles/r06_ee_ddim.txt
"""
from __future__ import annotations

import argparse
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tools.bench_dpm_solver import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", type=Path, required=True)
    ap.add_argument("--batch", type=int, default=128)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ee_ddim needs a B200: there is no CPU measurement")
    import bench
    import duodiff_b200 as ddb
    from duodiff_b200 import eesampler as ES
    from duodiff_b200.configs import CONFIGS
    from duodiff_b200.ddpm import Sampler
    from duodiff_b200.sampler import _ddim_plan

    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card (name, power.limit, clocks.max.sm): {card()}")
    dev = torch.device("cuda:0")
    B = args.batch
    _, full, _ = bench.PAIRS["celeba"]
    pf = CONFIGS[full]
    depth, C, H = pf["depth"], pf["in_chans"], pf["img_size"]
    torch.manual_seed(1234)
    net = ddb.EarlyExitUViT(ddb.UViT(**pf, max_batch=B), "mlp_probe_per_layer")
    bench.synthetic_probes_(net, depth, 1.0, 0.5)
    net = net.eval().to(dev)
    eng = net.engine(B)
    x_T = torch.randn(B, C, H, H, device=dev, generator=torch.Generator(device=dev).manual_seed(1000))
    log(f"CelebA deediff (depth {depth}), mlp_probe_per_layer with synthetic probes (slope 1.0, wscale 0.5), "
        f"random-init weights, B = {B}, compaction mode (ee_mode 1), DDIM eta 0")
    samplers = (("DDPM 1000", None), ("DDIM 100", 100), ("DDIM 50", 50))
    idx_logs = {}
    for thr in (0.08, 0.0):
        for label, n in samplers:
            kw = dict(seed=0, num_channels=C, sample_height=H, sample_width=H, threshold=thr, depth=depth, mode=1)
            if n is not None:
                kw.update(use_ddim=True, ddim_steps=n)
            ES.get_samples(net, B, **kw)  # warm-up: graphs captured, sampler cached
            torch.cuda.synchronize()
            rates = []
            for _ in range(2):
                tic = time.perf_counter()
                out, _err, idx = ES.get_samples(net, B, **kw)
                torch.cuda.synchronize()
                rates.append(B / (time.perf_counter() - tic))
            visited = ~torch.isnan(idx[:, 0])
            idx_logs[(thr, label)] = idx
            # in-graph step time: whole replayed trajectories on a sampler of the same rule
            rule = ("ddim", n, 0.0) if n is not None else "predict_noise"
            smp = Sampler(eng, None, np.inf, B, rule=rule, ee_threshold=thr, ee_mode=1)
            steps, flags = _ddim_plan(n, False, np.inf) if n is not None else (list(range(999, -1, -1)), [False] * 1000)
            smp.run_list(x_T.clone(), steps, flags, seed=1)
            ms = []
            for rep in range(3):
                x = x_T.clone()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                smp.run_list(x, steps, flags, seed=2 + rep)
                b.record()
                torch.cuda.synchronize()
                ms.append(a.elapsed_time(b) / len(steps))
            del smp
            log(f"threshold {thr:.2f}, {label:9s} ({int(visited.sum()):4d} model evaluations): "
                f"{max(rates):7.2f} images/s (of 2 runs: {min(rates):.2f}..{max(rates):.2f}); in-graph "
                f"{min(ms):.3f} ms/step (of 3: {min(ms):.3f}..{max(ms):.3f}); mean exit layer "
                f"{idx[visited].mean().item():.2f} of {depth}; samples finite: {bool(np.isfinite(out).all())}")
    # do the probes exit at the same layers on the DDIM grid as on the 1000-step trajectory at those timesteps?
    ddpm = idx_logs[(0.08, "DDPM 1000")]
    log("mean exit layer per timestep band, threshold 0.08: DDPM 1000 at the DDIM grid's timesteps vs the DDIM run")
    for label, n in samplers[1:]:
        grid = _ddim_plan(n, False, np.inf)[0]
        ddim = idx_logs[(0.08, label)]
        bands = []
        for lo, hi in ((700, 1000), (300, 700), (0, 300)):
            rows = [t for t in grid if lo <= t < hi]
            bands.append(f"t in [{lo}, {hi}): {ddpm[rows].mean().item():.2f} vs {ddim[rows].mean().item():.2f}")
        same = (ddpm[grid] == ddim[grid]).float().mean().item()
        log(f"  {label}: all grid steps {ddpm[grid].mean().item():.2f} vs {ddim[grid].mean().item():.2f}; "
            + "; ".join(bands) + f"; same exit layer for {100 * same:.1f} % of (t, sample)")
    log("FID: not measured (the Inception weights are not available)")
    log(f"card after the runs: {card()}")
    args.out.parent.mkdir(parents=True, exist_ok=True)
    args.out.write_text("# python tools/bench_ee_ddim.py (one B200)\n" + "\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
