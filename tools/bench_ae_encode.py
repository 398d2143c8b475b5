"""Throughput of the KL-autoencoder encoder (FrozenAutoencoderKL.encode_moments) on get_autoencoder's ddconfig.

    python tools/bench_ae_encode.py [--batch 64] [--chunk 32] [--iters 20] [--no-oracle]

Random-init weights (random_init_state_dict(encoder=True)), images uniform in [-1, 1], B images in chunks of
`--chunk` (decode's measurement setup), warm-up, CUDA events.  Reports ms per image, algorithmic TFLOP/s
(272.7 GFLOP / image, quant_conv not counted), the per-category split of ddb_ae_profile_encode (a separate run with an
event around every launch), and the card name and power limit read in the same run.  For context only: the same
encoder through oracle/ae_encoder_oracle.py on the GPU under bf16 autocast (cuDNN convolutions).
"""
import argparse
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from duodiff_b200.autoencoder import DEFAULT_DDCONFIG, FrozenAutoencoderKL, random_init_state_dict  # noqa: E402
from oracle import ae_encoder_oracle as E  # noqa: E402

GFLOP_PER_IMAGE = 272.7


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--chunk", type=int, default=32)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--no-oracle", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_ae_encode: needs a CUDA device (no CPU measurement)")
    print(f"card: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, clocks.max.sm: {card()}")
    sd = random_init_state_dict(DEFAULT_DDCONFIG, 4, 0, encoder=True)
    ae = FrozenAutoencoderKL(DEFAULT_DDCONFIG, 4, state_dict=sd, max_batch=args.chunk)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(args.batch, 3, 256, 256, device="cuda", generator=g) * 2 - 1
    for _ in range(2):
        ae.encode_moments(x)
    torch.cuda.synchronize()
    ms = timed(lambda: ae.encode_moments(x), args.iters)
    tf = GFLOP_PER_IMAGE * args.batch / ms  # GFLOP / ms = TFLOP/s
    print(f"encode_moments B={args.batch} chunk={args.chunk}: {ms:.2f} ms  ({ms / args.batch:.3f} ms/img, "
          f"{1000 * args.batch / ms:.1f} img/s, {tf:.1f} TFLOP/s algorithmic at {GFLOP_PER_IMAGE} GFLOP/img)")
    z_ms = timed(lambda: ae.encode(x), args.iters) - ms
    print(f"  encode = encode_moments + sample (randn_like + ddb_ae_sample): +{z_ms:.3f} ms for the batch")
    prof = ae.profile_encode(x)
    tot_ms = sum(v["ms"] for v in prof.values())
    tot_f = sum(v["flops"] for v in prof.values())
    print(f"profile_encode (event around every launch): {tot_ms:.2f} ms, {tot_f / args.batch / 1e9:.1f} GFLOP/img")
    for k, v in prof.items():
        rate = v["flops"] / v["ms"] / 1e9 if v["ms"] > 0 and v["flops"] > 0 else 0.0
        print(f"    {k:14s} {v['ms']:8.3f} ms  {100 * v['ms'] / tot_ms:5.1f} %  {rate:7.1f} TFLOP/s")
    if args.no_oracle:
        return
    del ae
    torch.cuda.empty_cache()
    spec = E.AEEncSpec()
    sdc = {k: v.cuda() for k, v in sd.items() if k.startswith(("encoder.", "quant_conv."))}
    xs = x[:args.chunk]

    def ref():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            E.encode_moments(sdc, spec, xs)
    torch.backends.cudnn.benchmark = True
    for _ in range(2):
        ref()
    torch.cuda.synchronize()
    rms = timed(ref, args.iters)
    print(f"context: oracle encode_moments under bf16 autocast (cuDNN), B={args.chunk}: {rms:.2f} ms "
          f"({rms / args.chunk:.3f} ms/img, {GFLOP_PER_IMAGE * args.chunk / rms:.1f} TFLOP/s algorithmic)")


if __name__ == "__main__":
    main()
