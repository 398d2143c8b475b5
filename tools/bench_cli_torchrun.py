"""Images/s of the `sampler.py` command line itself, alone and under `torchrun --standalone --nproc-per-node N`.

    python tools/bench_cli_torchrun.py [--per-gpu 128] [--out report.txt]

Writes random-init checkpoints and yaml configs to a temporary directory and runs, from the repository root:
  * the CelebA DuoDiff pair (celeba_3 -> celeba, --t_switch 300, 1000 DDPM steps), B = --per-gpu images per GPU, for
    every N of 1, 2 and 8 that the visible GPUs allow (one GPU per rank);
  * the ImageNet-256 latent pair (imagenet256_3 -> imagenet256, --class_id, the KL-autoencoder decode to 256x256x3 inside
    the timed region) at the largest of those N, and -- when that N is 1 -- also 2 ranks sharing the one GPU, so that
    the gloo gather of the decoded images is measured (its throughput is then not a scaling figure).
images/s = global batch / the `Elapsed time` of statistics.txt (model loading excluded, the gather included); the
gather's time is the line rank 0 prints.  The card's name and power limit are read in the same run.  An N that was
not run is reported as "not measured".  Command lines are logged with the temporary directory written as $TMP.
"""
import argparse
import os
import re
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import torch
import yaml

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import duodiff_b200 as ddb  # noqa: E402
from duodiff_b200.configs import CONFIGS  # noqa: E402
from tests.process_tree import run_tree  # noqa: E402

TIMEOUT = 3000


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def write_model(tmp: Path, name: str, seed: int, extra_cfg=None):
    torch.manual_seed(seed)
    ck, cfg = tmp / f"{name}.pth", tmp / f"{name}.yaml"
    torch.save(ddb.UViT(**CONFIGS[name]).state_dict(), ck)
    c = {"model_params": dict(CONFIGS[name]), "dataset": "synthetic"}
    c.update(extra_cfg or {})
    cfg.write_text(yaml.safe_dump(c))
    return str(ck), str(cfg)


def run(label, nproc, args, out: Path, log, env=None):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(nproc), "sampler.py",
           *args, "--output_folder", str(out)]
    t0 = time.time()
    rc, output = run_tree(cmd, TIMEOUT, cwd=ROOT, env=env)  # on timeout no rank is left running
    wall = time.time() - t0
    if rc != 0:
        why = f"timed out after {TIMEOUT} s" if rc is None else f"exit {rc}"
        log(f"{label}: FAILED ({why})\n{output[-3000:]}")
        return
    elapsed = float((out / "statistics.txt").read_text().split()[2])
    m = re.search(r"Gathered (\d+) samples from (\d+) ranks in ([0-9.]+) s", output)
    gather = f"gather {float(m.group(3)):.3f} s = {100 * float(m.group(3)) / elapsed:.2f} % of elapsed" if m \
        else "no gather (one process)"
    G = int(args[args.index("--batch_size") + 1])
    log(f"{label}: G = {G}, Elapsed time {elapsed:.3f} s -> {G / elapsed:.2f} images/s "
        f"({G / elapsed / nproc:.2f} per rank); {gather}; process wall time incl. start-up and PNGs "
        f"{wall:.1f} s")
    log("    " + " ".join(cmd[1:]).replace(str(out.parent), "$TMP"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-gpu", type=int, default=128)
    ap.add_argument("--out", type=str, default=None, help="also write the report to this file")
    a = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    n_gpu = torch.cuda.device_count()
    log(f"card (nvidia-smi index, name, power.limit): {card()}")
    log(f"visible GPUs: {n_gpu}; B = {a.per_gpu} per GPU; random-init weights, seed 0")
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        ck_e, cfg_e = write_model(tmp, "celeba_3", 1)
        ck_l, cfg_l = write_model(tmp, "celeba", 2)
        ns = [n for n in (1, 2, 8) if n <= n_gpu]
        for n in (1, 2, 8):
            if n not in ns:
                log(f"CelebA DuoDiff N = {n}: not measured ({n_gpu} GPU(s) visible)")
                continue
            G = a.per_gpu * n
            args = ["--checkpoint_path", ck_e, "--config_path", cfg_e, "--checkpoint_path_late", ck_l,
                    "--config_path_late", cfg_l, "--t_switch", "300", "--batch_size", str(G), "--parametrization",
                    "predict_noise"]
            run(f"CelebA DuoDiff N = {n}", n, args, tmp / f"celeba_n{n}", log)
        from oracle.ae_oracle import AESpec, random_state_dict
        ae = tmp / "ae.pth"
        torch.save(random_state_dict(AESpec(), 3), ae)
        extra = {"autoencoder": {"autoencoder_checkpoint_path": str(ae)}}
        ck_e, cfg_e = write_model(tmp, "imagenet256_3", 4, extra)
        ck_l, cfg_l = write_model(tmp, "imagenet256", 5, extra)
        n = max(ns)
        cases = [(f"ImageNet-256 + decode N = {n}", n, None)]
        if n == 1:
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            cases.append(("ImageNet-256 + decode, 2 ranks sharing one GPU", 2,
                          dict(os.environ, CUDA_VISIBLE_DEVICES=visible.split(",")[0] if visible else "0")))
        for label, nproc, env in cases:
            G = a.per_gpu * (n if env is None else 1)
            args = ["--checkpoint_path", ck_e, "--config_path", cfg_e, "--checkpoint_path_late", ck_l,
                    "--config_path_late", cfg_l, "--t_switch", "300", "--batch_size", str(G), "--parametrization",
                    "predict_noise", "--class_id", "1"]
            run(label, nproc, args, tmp / f"in256_{nproc}_{env is None}", log, env)
    log(f"card after the runs: {card()}")
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
