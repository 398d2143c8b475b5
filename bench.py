#!/usr/bin/env python
"""bench.py — DuoDiff sampling throughput (images/sec, 1000 DDPM steps, t_switch=300) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config celeba] [--batch 128]
                    [--ee [--threshold 0.08] [--slope 0.5]] [--decode] [--verify-shards] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: a full 1000-step DuoDiff sampling of `batch` images per GPU
(300 shallow-U-ViT steps, 700 full-U-ViT steps, 1000 DDPM updates).  One JSON line on stdout (rank 0):
  value  = whole-job images/sec with x_T already resident in HBM, CUDA-event timed, max over ranks
  e2e    = the same through the public API duodiff_b200.sampler.get_samples(): x_T drawn on the host, pinned
           H2D copy, 1000 steps, (x+1)/2 NHWC, D2H to numpy — all inside the timed region
  roofline / kernels = per-kernel CUDA-event timings of one shallow + one full sampling STEP as the sampler runs it
           (ddb_sampler_profile_step, eager), tensor-bound categories as TFLOP/s vs the sustained bf16 peak,
           memory-bound ones as GB/s vs the measured HBM copy bandwidth; `step_ms_in_graph` = the same steps timed as
           CUDA-graph replays, which is what `ms_per_step` is made of (eager event pairs lose the PDL overlap)
  cpu_baseline = the UNMODIFIED reference (baseline/_ref) on the host cores, bounded sample, rank 0, N=1 only
`--impl reference` times the reference's own CPU implementation of the path instead (see DESIGN.md §5).
`--ee` measures BASELINE config 3 (DeeDiff early exit, compaction mode) instead of the DuoDiff pair.
`--verify-shards` is a correctness run, not a benchmark: N-rank sharded sampling == single-GPU sampling row for row.
`--dump-outputs DIR` writes what the timed path returned in its last timed step as DIR/<name>.npy (see dump_outputs):
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

from duodiff_b200.configs import CONFIGS  # noqa: E402

PAIRS = {  # BASELINE.json configs -> (shallow, full, default batch per GPU)
    "cifar10": ("cifar10_3", "cifar10", 128),
    "celeba": ("celeba_3", "celeba", 128),
    "imagenet64": ("imagenet64_3", "imagenet64", 256),
    "imagenet256": ("imagenet256_3", "imagenet256", 256),
}
T_SWITCH = 300
METRIC = "images/sec (DuoDiff sampling, 1000 steps)"
METRIC_EE = "images/sec (DeeDiff early-exit sampling, 1000 steps)"


def forward_flops(p: dict) -> dict:
    """Algorithmic FLOPs per image per forward (SURVEY.md §8d), split per kernel category."""
    D, d = p["embed_dim"], p["depth"]
    N = (p["img_size"] // p["patch_size"]) ** 2
    L = N + (2 if p["num_classes"] > 0 else 1)
    pd = p["patch_size"] ** 2 * p["in_chans"]
    hid = int(D * p["mlp_ratio"])
    per = dict(gemm_qkv=d * 2 * L * D * 3 * D, gemm_proj=d * 2 * L * D * D, gemm_fc1=d * 2 * L * D * hid,
               gemm_fc2=d * 2 * L * hid * D, gemm_skip=(d // 2) * 2 * L * 2 * D * D, attention=d * 4 * L * L * D,
               gemm_decode=2 * L * D * pd, embed=2 * N * pd * D,
               conv=18 * p["in_chans"] ** 2 * p["img_size"] ** 2)
    per["total"] = sum(per.values())
    return per


def block_flops(p: dict, i: int) -> int:
    """FLOPs per image of block i alone (long-skip GEMM included for the out-blocks)."""
    D, d = p["embed_dim"], p["depth"]
    L = (p["img_size"] // p["patch_size"]) ** 2 + (2 if p["num_classes"] > 0 else 1)
    f = 24 * L * D * D + 4 * L * L * D
    return f + (4 * L * D * D if i > d // 2 else 0)


def launch_bytes(p: dict, B: int) -> dict:
    """ALGORITHMIC HBM bytes per launch of the memory-bound categories (SURVEY.md §8d): every tensor the kernel must
    read or write once, nothing for re-reads, weights or L2 hits."""
    D = p["embed_dim"]
    N = (p["img_size"] // p["patch_size"]) ** 2
    L = N + (2 if p["num_classes"] > 0 else 1)
    n = B * p["in_chans"] * p["img_size"] ** 2
    M = B * L
    return dict(
        embed=B * N * 256 + M * D * 2,         # inside the sampler: read the bf16 hi|lo patch matrix, write the tokens
        attention=M * 3 * D * 2 + M * D * 2,   # q|k|v in, o out (bf16)
        gemm_decode=M * D * 2 + n * 4,         # tokens in (bf16), un-patchified image out (fp32)
        conv=2 * n * 4,                        # stand-alone 3x3 conv (early-exit heads)
        ddpm=3 * n * 4,                        # stand-alone update with in-kernel Philox: x, eps in; x out
        tail=3 * n * 4 + B * N * 256,          # fused: decoder image in, x in/out, next step's patch matrix out
        ln_stats=M * D * 2,                    # early exit: probe + LayerNorm statistics pass over the block input
    )


def peaks() -> dict:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return dict(tflops=d.get("bf16_tflops_sustained", d.get("bf16_tflops")), tflops_burst=d.get("bf16_tflops"),
                    hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def workload_config(name: str, B: int, world: int, extra: str = "") -> dict:
    """The `config` object of the JSON line: identical for the GPU arm and the reference arm of the same workload."""
    shallow, full, _ = PAIRS[name]
    return dict(workload=f"DuoDiff {name} ({shallow}+{full}) 1000 DDPM steps, t_switch={T_SWITCH}" + extra,
                batch_per_gpu=B, global_batch=B * world, t_switch=T_SWITCH, parallelism=f"dp{world}",
                l2="no flush: one DDPM step touches ~1 GB of activations+weights (> 126 MB L2)")


DUMP_LIMIT = 64 << 20  # bytes of .npy data per --dump-outputs directory


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each array as out_dir/<name>.npy in float32 (integer logs converted), at most DUMP_LIMIT bytes in all.
    Smaller arrays are written whole; one that does not fit its share of what is left is replaced by a fixed sample of
    its rows (leading dimension, seed 0, kept in order), so that the same arguments always select the same rows."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    items = sorted(((k, v.detach().float().cpu().numpy()) for k, v in arrays.items()), key=lambda kv: kv[1].nbytes)
    left = DUMP_LIMIT
    for i, (name, a) in enumerate(items):
        share = left // (len(items) - i) - 4096  # headroom for the .npy header
        if a.nbytes > share:
            keep = share // a[0].nbytes
            if keep < 1:
                raise ValueError(f"--dump-outputs: one row of {name} {a.shape} exceeds {share} bytes")
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(d / f"{name}.npy", a)
        left -= (d / f"{name}.npy").stat().st_size


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self) -> dict:
        sm, mx, reasons, power, watts = [], 0, set(), 0.0, []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                power = max(power, float(r[6]))
                watts.append(float(r[6]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        busy = [c for c in sm if c > 0]
        return dict(sm_mhz=statistics.median(busy) if busy else None, sm_max_mhz=mx or None,
                    reasons=sorted(reasons), power_w_max=power or None,
                    power_w_median=statistics.median(watts) if watts else None, samples=len(sm))


# ------------------------------------------------------------------------------------------------ reference (CPU) arm
def _load_reference():
    """The UNMODIFIED reference modules staged under baseline/_ref (git-ignored; travels with gpurun): its `sampler`
    module (get_samples, predict_noise_postprocessing, the module-level schedule) and `models.uvit.UViT`.  matplotlib
    (only used by dump_samples) is stubbed.  Returns None when the copy is absent -> the oracle port is timed."""
    import importlib.util
    import types
    ref = ROOT / "baseline" / "_ref"
    if not (ref / "sampler.py").exists() or not (ref / "models" / "uvit.py").exists():
        return None
    mpl, pp = types.ModuleType("matplotlib"), types.ModuleType("matplotlib.pyplot")
    mpl.pyplot = pp
    sys.modules.setdefault("matplotlib", mpl)
    sys.modules.setdefault("matplotlib.pyplot", pp)
    sys.path.insert(0, str(ref))  # the reference imports `models.*` / `utils.*` as top-level packages
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            spec = importlib.util.spec_from_file_location("_duodiff_reference_sampler", ref / "sampler.py")
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
        return mod
    except Exception as e:  # noqa: BLE001
        print(f"[bench] reference import failed ({e!r}); timing the oracle port instead", file=sys.stderr)
        return None
    finally:
        sys.path.remove(str(ref))


def run_reference(args, rank: int, world: int) -> None:
    """The reference's CPU implementation of the path on this box's host cores (all threads).  One `step` = a bounded
    sample of the workload AT THE CONFIGURED BATCH: 1 shallow-backbone forward + 1 full-backbone forward + 2 DDPM
    updates through the reference's own predict_noise_postprocessing (sampler.py:47-56); value = batch / (300 t_shallow
    + 700 t_full + 1000 t_update) from the medians over the timed steps.  --full-run executes the unmodified
    sampler.get_samples for all 1000 steps instead (BASELINE config 1: CIFAR-10, batch 8)."""
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    torch.set_num_threads(max(1, os.cpu_count() or 1))  # torchrun exports OMP_NUM_THREADS=1
    shallow, full, default_b = PAIRS[args.config]
    B = args.batch or default_b
    ps, pf = CONFIGS[shallow], CONFIGS[full]
    ref = _load_reference()
    kind = "reference" if ref is not None else "port"
    torch.manual_seed(1234)
    if ref is not None:
        with contextlib.redirect_stdout(io.StringIO()):
            nets = {shallow: ref.UViT(**ps).eval(), full: ref.UViT(**pf).eval()}
        fwd = {k: (lambda mm: (lambda x, t, y: mm(x, t, y)))(m) for k, m in nets.items()}
        update = ref.predict_noise_postprocessing  # draws z with torch.randn_like like the reference does
    else:
        import duodiff_b200 as ddb
        from oracle import uvit_oracle as O
        fwd = {}
        for name, p in ((shallow, ps), (full, pf)):
            sd, spec = ddb.UViT(**p).state_dict(), O.UViTSpec.from_params(p)
            fwd[name] = (lambda s, sp: (lambda x, t, y: O.uvit_forward(s, sp, x, t, y)))(sd, spec)
        sch = O.ddpm_schedule()
        update = lambda eps, x, t: O.predict_noise_step(sch, eps, x, t, torch.randn_like(x))  # noqa: E731
    C, H = pf["in_chans"], pf["img_size"]
    y = torch.randint(0, min(ps["num_classes"], pf["num_classes"]), (B,)) if pf["num_classes"] > 0 else None
    t_begin = time.perf_counter()
    if args.full_run:
        if ref is None:
            raise SystemExit("--full-run needs the reference copy under baseline/_ref")
        vals = []
        for i in range(warm + steps):
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                out, _ = ref.get_samples(model=nets[shallow], batch_size=B, postprocessing=update, seed=i,
                                         num_channels=C, sample_height=H, sample_width=H, use_ddim=False,
                                         ddim_steps=50, ddim_eta=0.0, timesteps_save=[], y=y, autoencoder=None,
                                         late_model=nets[full], t_switch=T_SWITCH)
            dt = time.perf_counter() - t0
            assert out.shape == (B, H, H, C)
            if i >= warm:
                vals.append(B / dt)
        v, sample = statistics.median(vals), (f"{len(vals)} x the unmodified sampler.get_samples, all 1000 steps "
                                              f"({T_SWITCH} {shallow} + {1000 - T_SWITCH} {full}) at batch {B}, fp32")
        extra = dict(values=vals)
    else:
        x = torch.randn(B, C, H, H)
        times = {shallow: [], full: [], "update": []}
        with torch.no_grad():
            for i in range(warm + steps):
                for name, t in ((shallow, 800), (full, 400)):
                    tt = t * torch.ones(B)
                    t0 = time.perf_counter()
                    eps = fwd[name](x, tt, y)
                    t1 = time.perf_counter()
                    x = update(eps, x, t)
                    t2 = time.perf_counter()
                    if i >= warm:
                        times[name].append(t1 - t0)
                        times["update"].append(t2 - t1)
                x = x.clamp(-3, 3)  # the bounded sample repeats two timesteps: keep x in the range of real iterates
        med = {k: statistics.median(v) for k, v in times.items()}
        mn = {k: min(v) for k, v in times.items()}
        total = lambda d: T_SWITCH * d[shallow] + (1000 - T_SWITCH) * d[full] + 1000 * d["update"]  # noqa: E731
        v = B / total(med)
        sample = (f"{steps} x (1 {shallow} fwd + 1 {full} fwd + 2 DDPM updates via the reference's "
                  f"predict_noise_postprocessing) at batch {B}, fp32; medians t_shallow={med[shallow]:.3f}s "
                  f"t_full={med[full]:.3f}s t_update={med['update']:.4f}s extrapolated to {T_SWITCH}+{1000 - T_SWITCH} steps")
        extra = dict(value_from_min=B / total(mn), value_from_median=v, reps=steps)
    ms = (time.perf_counter() - t_begin) * 1e3 / (warm + steps)
    info = dict(value=v, unit="images/sec", cores=torch.get_num_threads(), kind=kind, sample=sample,
                host_cpus=os.cpu_count(), **extra)
    line = dict(impl="reference", metric=METRIC, value=v, unit="images/sec", n_gpus=args.gpus, steps=steps,
                warmup=warm, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic (random-init weights, N(0,1) x_T)", config=workload_config(args.config, B, args.gpus),
                cpu_baseline=info, e2e=dict(value=v, unit="images/sec", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0,
                note=("N > 1: one CPU process on rank 0 only; dividing an N-GPU value by it multiplies the 1-GPU "
                      "ratio by N" if args.gpus > 1 else None))
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(args, B: int) -> dict | None:
    """The reference arm as a child process with the GPU hidden (this process has CUDA initialised; the reference's
    module-level `device = get_device()` must resolve to the CPU)."""
    cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--config", args.config, "--batch", str(B),
           "--steps", "3", "--warmup", "1"]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMP_NUM_THREADS"):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return dict(error=(r.stderr or r.stdout)[-400:])
    except Exception as e:  # noqa: BLE001
        return dict(error=repr(e))


# ------------------------------------------------------------------------------------------------ GPU arm
def _kernel_table(prof_fn, fl: dict | None, nbytes: dict, B: int, pk: dict, reps: int = 5) -> dict:
    """Average `reps` eager profiled steps; per category: ms, launches, share, TFLOP/s (tensor-bound categories) or
    GB/s + fraction of the measured HBM bandwidth (memory-bound categories, algorithmic bytes)."""
    for _ in range(2):
        prof = prof_fn()
    acc = {k: 0.0 for k in prof}
    for _ in range(reps):
        prof = prof_fn()
        for k, v in prof.items():
            acc[k] += v["ms"] / reps
    tot = sum(acc.values())
    table = {}
    for k in acc:
        n = prof[k]["launches"]
        if not n:
            continue
        row = dict(ms=round(acc[k], 4), launches=n, share=round(acc[k] / tot, 4))
        if fl and k in fl and k.startswith(("gemm_q", "gemm_p", "gemm_f", "gemm_s", "attention")):
            row["tflops"] = round(fl[k] * B / (acc[k] * 1e-3) / 1e12, 1)
            row["frac_tensor"] = round(row["tflops"] / pk["tflops"], 4)
        if k in nbytes:
            gbps = nbytes[k] * n / (acc[k] * 1e-3) / 1e9
            row["gbps"] = round(gbps, 1)
            row["frac_hbm"] = round(gbps / pk["hbm"], 4)
            row["bytes_per_launch"] = nbytes[k]
        table[k] = row
    table["_step_ms_sum_eager"] = round(tot, 4)
    return table


def _time_steps(smp, x, y, t_first: int, n: int) -> float:
    """ms per step of `n` graph-replayed sampling steps starting at t_first (CUDA events on the launching stream)."""
    smp.run(x, y=y, seed=1, t_first=t_first, t_last=t_first - n + 1, use_graph=True)  # capture / warm
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    smp.run(x, y=y, seed=1, t_first=t_first, t_last=t_first - n + 1, use_graph=True)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def run_ours(args, rank: int, world: int, local_rank: int) -> None:
    import torch.distributed as dist

    import duodiff_b200 as ddb
    from duodiff_b200 import _lib
    from duodiff_b200 import sampler as S
    from duodiff_b200.ddpm import Sampler

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    shallow, full, default_b = PAIRS[args.config]
    B = args.batch or default_b
    ps, pf = CONFIGS[shallow], CONFIGS[full]
    torch.manual_seed(1234)  # identical random-init weights on every rank (SURVEY.md §8d C2)
    early = ddb.UViT(**ps, max_batch=B).eval().to(dev)
    late = ddb.UViT(**pf, max_batch=B).eval().to(dev)
    C, H = pf["in_chans"], pf["img_size"]
    y = None
    if pf["num_classes"] > 0:
        y = torch.randint(0, min(ps["num_classes"], pf["num_classes"]), (B,), device=dev)
    lib = _lib.load()
    ae = None
    if args.decode:  # latent configs: KL-autoencoder decode after the loop (sampler.py:141-143), random-init weights
        from duodiff_b200 import autoencoder as AE
        assert C == 4 and H == 32, "--decode needs a latent config (imagenet256)"
        with contextlib.redirect_stdout(sys.stderr):  # the shim prints like the reference; stdout carries the JSON line
            ae = AE.FrozenAutoencoderKL(AE.DEFAULT_DDCONFIG, 4, state_dict=AE.random_init_state_dict(seed=4321),
                                        max_batch=min(B, 32))
    smp = Sampler(early.engine(B), late.engine(B), T_SWITCH, B)
    smp.set_noise_offset(rank * B)  # rows [rank*B, (rank+1)*B) of the global batch
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    n_total = args.warmup + args.steps
    x_all = [torch.randn(B, C, H, H, device=dev, generator=gen) for _ in range(min(n_total, 4))]
    oshape = (B, 256, 256, 3) if ae is not None else (B, H, H, C)
    gathered = [torch.empty(*oshape, device=dev) for _ in range(world)] if world > 1 else None

    def one_pass(i: int):
        x = x_all[i % len(x_all)].clone()
        smp.run(x, y=y, seed=i, use_graph=True)
        out = smp.finalize(ae.decode(x) if ae is not None else x)
        if world > 1:
            dist.all_gather(gathered, out)  # the path's only collective: finished samples (SURVEY.md §8e)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident-input throughput (value)
    for i in range(args.warmup):
        one_pass(i)
    barrier()
    l0 = lib.ddb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        e0.record()
        for i in range(args.steps):
            out = one_pass(args.warmup + i)
        e1.record()
        barrier()
    launches = lib.ddb_launch_count() - l0
    ms = e0.elapsed_time(e1)
    assert torch.isfinite(out).all(), "non-finite samples"
    if args.dump_outputs and rank == 0:  # the finished samples of the whole job, [world*B, H, W, C] (NHWC, in [0, 1])
        dump_outputs(args.dump_outputs, dict(samples=torch.cat(gathered) if world > 1 else out))

    # ---- end-to-end through the public API (host x_T -> H2D -> 1000 steps -> NHWC -> D2H numpy)
    def e2e_pass(i: int):
        with contextlib.redirect_stdout(sys.stderr):
            return S.get_samples(early, B, S.predict_noise_postprocessing, seed=i, num_channels=C, sample_height=H,
                                 sample_width=H, use_ddim=False, ddim_steps=50, ddim_eta=0.0, timesteps_save=[], y=y,
                                 autoencoder=ae, late_model=late, t_switch=T_SWITCH, device=dev,
                                 noise_row_offset=rank * B)[0]

    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    for i in range(min(args.warmup, 1)):
        e2e_pass(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        host = e2e_pass(100 + i)
    barrier()
    e2e_s = time.perf_counter() - t0
    assert host.shape == oshape

    # ---- reduce over ranks (max time)
    tt = torch.tensor([ms, e2e_s * 1e3, float(launches)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max = tt[0].item(), tt[1].item()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * B * args.steps / (ms_max / 1e3)
    e2e_val = world * B * e2e_steps / (e2e_ms_max / 1e3)
    pk = peaks()
    fl_s, fl_f = forward_flops(ps), forward_flops(pf)
    flops_per_image = T_SWITCH * fl_s["total"] + (1000 - T_SWITCH) * fl_f["total"]

    # ---- per-kernel roofline: one eager sampling step per backbone with a CUDA-event pair around every launch
    xs = x_all[0].clone()
    kernels = {
        shallow: _kernel_table(lambda: smp.profile_step(xs, 800, False, y), fl_s, launch_bytes(ps, B), B, pk),
        full: _kernel_table(lambda: smp.profile_step(xs, 400, True, y), fl_f, launch_bytes(pf, B), B, pk),
    }
    # the same steps as CUDA-graph replays (PDL overlap kept): what ms_per_step is made of
    g_s = _time_steps(smp, x_all[0].clone(), y, 999, 50)
    g_f = _time_steps(smp, x_all[0].clone(), y, 500, 50)
    step_in_graph = dict(shallow_ms=round(g_s, 4), full_ms=round(g_f, 4),
                         pass_ms_from_steps=round(T_SWITCH * g_s + (1000 - T_SWITCH) * g_f, 1),
                         pass_ms_measured=round(ms_max / args.steps, 1),
                         eager_event_sum_ms=round(T_SWITCH * kernels[shallow]["_step_ms_sum_eager"]
                                                  + (1000 - T_SWITCH) * kernels[full]["_step_ms_sum_eager"], 1),
                         note="eager event pairs serialise the kernels (no programmatic-dependent-launch overlap): the "
                              "per-kernel TFLOP/s and GB/s below are pessimistic by eager_event_sum / pass_ms_from_steps")
    kf = kernels[full]
    # the north star's "fraction of bf16 tensor-core peak on the U-ViT GEMMs": GEMM FLOPs / summed GEMM-kernel time
    gk = [k for k in kf if k.startswith("gemm_") and k != "gemm_decode"]
    gemm_tf = sum(fl_f[k] for k in gk) * B / (sum(kf[k]["ms"] for k in gk) * 1e-3) / 1e12
    scale = step_in_graph["eager_event_sum_ms"] / step_in_graph["pass_ms_from_steps"]
    gemm_only = dict(tflops=round(gemm_tf, 1), frac_of_sustained_peak=round(gemm_tf / pk["tflops"], 4),
                     frac_of_burst_peak=round(gemm_tf / pk["tflops_burst"], 4) if pk.get("tflops_burst") else None,
                     in_graph_estimate_tflops=round(gemm_tf * scale, 1),
                     in_graph_estimate_frac_of_sustained=round(gemm_tf * scale / pk["tflops"], 4), kernels=gk)
    dom = max((k for k in kf if not k.startswith("_")), key=lambda k: kf[k]["ms"])
    dom_ms = kf[dom]["ms"] / kf[dom]["launches"]
    dom_flops = fl_f[dom] * B / kf[dom]["launches"]
    achieved = dom_flops / (dom_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    tf = ROOT / "profiles" / "traffic.json"
    if tf.exists():
        tj = json.loads(tf.read_text())
        traffic, traffic_src = tj.get(dom), tj.get("_source")
    roofline = dict(bound="tensor", kernel=f"{dom} (gemm2_tcgen05_kernel, CTA pair)" if dom.startswith("gemm") else dom,
                    achieved=round(achieved, 1), peak=pk["tflops"], unit="TFLOP/s", frac=round(achieved / pk["tflops"], 4),
                    traffic=traffic, traffic_provenance=("NOT measured in this run: " + traffic_src) if traffic_src else None,
                    peak_source=pk["source"] + ", sustained bf16; memory-bound kernels vs hbm_gbs copy bandwidth",
                    flops_per_launch=dom_flops, avg_launch_ms=round(dom_ms, 4),
                    gemm_only=gemm_only, hbm_peak_gbs=pk["hbm"],
                    whole_path=dict(tflops=round(value * flops_per_image / 1e12, 1),
                                    frac=round(value * flops_per_image / 1e12 / (pk["tflops"] * world), 4),
                                    flops_per_image=flops_per_image))

    cpu = cpu_baseline_subprocess(args, B) if world == 1 and not args.no_cpu else None
    nbytes = B * C * H * H * 4
    out_bytes = B * 256 * 256 * 3 * 4 if ae is not None else nbytes
    ae_info = None
    if ae is not None:  # per-category device time of one decode of the batch (CUDA events around every launch)
        prof = ae.profile_decode(x_all[0])
        ae_info = dict(ms_per_batch=round(sum(v["ms"] for v in prof.values()), 3),
                       gflop_per_image=round(sum(v["flops"] for v in prof.values()) / B / 1e9, 1),
                       categories={k: round(v["ms"], 3) for k, v in prof.items()})
    line = dict(metric=METRIC, value=round(value, 3), unit="images/sec", n_gpus=world, steps=args.steps,
                warmup=args.warmup, ms_per_step=round(ms_max / args.steps, 2), higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="bf16", data="synthetic (random-init weights, N(0,1) x_T, Philox z_t)",
                config=workload_config(args.config, B, world,
                                       " + KL-autoencoder decode to 3x256x256" if ae is not None else ""),
                clocks=clocks.summary(),
                e2e=dict(value=round(e2e_val, 3), unit="images/sec", h2d_bytes_per_step=nbytes,
                         d2h_bytes_per_step=out_bytes, steps=e2e_steps, api="duodiff_b200.sampler.get_samples"),
                gpu_launches=int(tt[2].item()), roofline=roofline, step_ms_in_graph=step_in_graph, kernels=kernels,
                cpu_baseline=cpu)
    if ae_info is not None:
        line["autoencoder"] = ae_info
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ early exit (config 3)
def synthetic_probes_(net, depth: int, slope: float, wscale: float = 0.5) -> None:
    """Random-init probes sit at 0.47..0.55 and never cross 0.08 (SURVEY.md §6, §8d C3): scale the probe weights by
    `wscale` (per-sample spread) and set bias_i = -slope * i so that the probe outputs fall with depth like a trained
    uncertainty estimator's; `slope` positions the mean exit layer.  Calibrated over the WHOLE 1000-step trajectory
    (tools/ee_calibrate.py, profiles/r02_ee_calibration.txt): with random-init backbones |x_t| grows to ~1e3 towards
    t = 0, so exits happen early at high t and late at low t; slope 1.0 / wscale 0.5 gives a mean exit layer of 8.9 of
    13 (0.68 x depth, the regime of the published DeeDiff trend: 12.6 / 17 at threshold 0.07)."""
    with torch.no_grad():
        for i in range(depth):
            net.matrix[f"{i}"].classifier[0].weight.mul_(wscale)
            net.matrix[f"{i}"].classifier[0].bias.fill_(-slope * i)


def run_ee(args, rank: int, world: int, local_rank: int) -> None:
    """BASELINE config 3: DeeDiff / AdaDiff early-exit sampling (deediff_<config>.yaml: the full backbone + one MLP
    probe and one output head per layer, threshold 0.08), exited samples compacted out of the batch."""
    import torch.distributed as dist

    import duodiff_b200 as ddb
    from duodiff_b200 import _lib
    from duodiff_b200 import eesampler as ES
    from duodiff_b200.ddpm import Sampler

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _, full, default_b = PAIRS[args.config]
    B = args.batch or default_b
    pf = CONFIGS[full]
    depth, C, H = pf["depth"], pf["in_chans"], pf["img_size"]
    torch.manual_seed(1234)
    net = ddb.EarlyExitUViT(ddb.UViT(**pf, max_batch=B), "mlp_probe_per_layer")
    synthetic_probes_(net, depth, args.slope, args.wscale)
    net = net.eval().to(dev)
    eng = net.engine(B)
    y = torch.randint(0, pf["num_classes"], (B,), device=dev) if pf["num_classes"] > 0 else None
    lib = _lib.load()
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    x0 = [torch.randn(B, C, H, H, device=dev, generator=gen) for _ in range(2)]
    exit_log = torch.zeros(1000, B, device=dev, dtype=torch.int32)
    score_log = torch.zeros(1000, depth, device=dev)
    samplers = {m: Sampler(eng, None, float("inf"), B, ee_threshold=thr, ee_mode=mode)
                for m, (thr, mode) in dict(compact=(args.threshold, 1), simulate=(args.threshold, 0),
                                           never_exit=(0.0, 1)).items()}
    plain = Sampler(eng, None, float("inf"), B)  # the same backbone without probes / heads
    for s in list(samplers.values()) + [plain]:
        s.set_noise_offset(rank * B)

    def one_pass(i: int, smp=samplers["compact"], t_last=0):
        x = x0[i % 2].clone()
        smp.run(x, y=y, seed=i, t_first=999, t_last=t_last, exit_log=exit_log if smp is not plain else None,
                score_log=score_log if smp is not plain else None, use_graph=True)
        return smp.finalize(x)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        one_pass(i)
    barrier()
    l0 = lib.ddb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        e0.record()
        for i in range(args.steps):
            out = one_pass(args.warmup + i)
        e1.record()
        barrier()
    launches = lib.ddb_launch_count() - l0
    ms = e0.elapsed_time(e1)
    assert torch.isfinite(out).all()
    if args.dump_outputs and rank == 0:  # rank 0's shard; the side measurements below overwrite both logs
        dump_outputs(args.dump_outputs, dict(samples=out, exit_log=exit_log, score_log=score_log))
    idx = exit_log.float()  # [1000, B] of the last pass
    mean_exit = idx.mean().item()
    exit_hist = torch.bincount(exit_log.flatten().long().cpu(), minlength=depth + 1).tolist()
    # FLOPs actually needed: blocks executed per sample = its exit index (depth = never left), + token assembly
    blocks = torch.tensor([block_flops(pf, i) for i in range(depth)], dtype=torch.float64)
    cum = torch.cat([torch.zeros(1, dtype=torch.float64), blocks.cumsum(0)]).to(dev)
    flops_pass = cum[exit_log.long()].sum().item()  # sum over (t, sample)

    # side measurements: simulate (reference semantics), never-exit (threshold 0) and the plain backbone
    side = {}
    # (whole 1000-step passes: the exit pattern depends on t)
    for name, smp in list(samplers.items()) + [("plain_backbone", plain)]:
        one_pass(0, smp, 950)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        one_pass(1, smp, 0)
        b.record()
        barrier()
        side[name + "_ms_per_step"] = round(a.elapsed_time(b) / 1000, 4)
    side["compact_speedup_over_simulate"] = round(side["simulate_ms_per_step"] / side["compact_ms_per_step"], 3)
    side["never_exit_overhead_vs_plain"] = round(side["never_exit_ms_per_step"] / side["plain_backbone_ms_per_step"] - 1, 4)

    def e2e_pass(i: int):
        with contextlib.redirect_stdout(sys.stderr):
            return ES.get_samples(net, B, seed=i, num_channels=C, sample_height=H, sample_width=H,
                                  threshold=args.threshold, depth=depth, y=y, mode=1, device=dev,
                                  noise_row_offset=rank * B)[0]

    e2e_pass(0)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    for i in range(e2e_steps):
        host = e2e_pass(100 + i)
    barrier()
    e2e_s = time.perf_counter() - t0
    assert host.shape == (B, H, H, C)
    tt = torch.tensor([ms, e2e_s * 1e3, float(launches)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    value = world * B * args.steps / (tt[0].item() / 1e3)
    achieved = flops_pass * args.steps / (ms / 1e3) / 1e12  # this rank's executed-block FLOPs
    prof = _kernel_table(lambda: samplers["compact"].profile_step(x0[0].clone(), 500, False, y), None,
                         launch_bytes(pf, B), B, pk)
    line = dict(metric=METRIC_EE, value=round(value, 3), unit="images/sec", n_gpus=world, steps=args.steps,
                warmup=args.warmup, ms_per_step=round(tt[0].item() / args.steps, 2), higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="bf16",
                data="synthetic (random-init weights; probe weights x4, bias_i = -slope*i so that exits occur)",
                config=dict(workload=f"DeeDiff {args.config} (deediff_{args.config}.yaml, mlp_probe_per_layer) 1000 DDPM "
                                     f"steps, threshold {args.threshold}, per-sample exit compaction",
                            batch_per_gpu=B, global_batch=B * world, threshold=args.threshold, probe_slope=args.slope,
                            probe_wscale=args.wscale,
                            parallelism=f"dp{world}",
                            l2="no flush: one DDPM step touches ~1 GB of activations+weights (> 126 MB L2)"),
                clocks=clocks.summary(),
                e2e=dict(value=round(world * B * e2e_steps / (tt[1].item() / 1e3), 3), unit="images/sec",
                         h2d_bytes_per_step=B * C * H * H * 4, d2h_bytes_per_step=B * C * H * H * 4, steps=e2e_steps,
                         api="duodiff_b200.eesampler.get_samples(mode=1)"),
                gpu_launches=int(tt[2].item()),
                early_exit=dict(mean_exit_layer=round(mean_exit, 3), depth=depth,
                                exit_histogram=exit_hist,
                                flops_executed_per_image=flops_pass / B, **side),
                roofline=dict(bound="tensor", kernel="executed blocks (sum of exit indices) of the compacted step",
                              achieved=round(achieved, 1), peak=pk["tflops"], unit="TFLOP/s",
                              frac=round(achieved / pk["tflops"], 4), traffic=None,
                              peak_source=pk["source"] + ", sustained bf16", hbm_peak_gbs=pk["hbm"]),
                kernels={"compact_step_t500": prof}, cpu_baseline=None)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ N-GPU correctness
def run_verify(args, rank: int, world: int, local_rank: int) -> None:
    """NCCL correctness, not speed (SURVEY.md §8e): the all-gathered result of N sharded ranks must equal rank 0's own
    single-GPU run of the GLOBAL batch, row for row -- DuoDiff with the hand-off inside the run (39 DDIM steps through
    the public get_samples API), once with injected noise and once with the seed-keyed Philox stream, plus the
    eesampler index / probe logs through duodiff_b200.distributed."""
    import numpy as np
    import torch.distributed as dist

    import duodiff_b200 as ddb
    from duodiff_b200 import distributed as D
    from duodiff_b200 import eesampler as ES
    from duodiff_b200 import sampler as S

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    shallow, full, _ = PAIRS[args.config]
    ps, pf = CONFIGS[shallow], CONFIGS[full]
    per = args.batch or 8
    G = per * world + (1 if world > 1 else 0)  # uneven shards
    C, H = pf["in_chans"], pf["img_size"]
    torch.manual_seed(1234)
    early = ddb.UViT(**ps, max_batch=G).eval().to(dev)
    late = ddb.UViT(**pf, max_batch=G).eval().to(dev)
    g = torch.Generator().manual_seed(99)
    noise = torch.randn(1000, G, C, H, H, generator=g)
    y = torch.randint(0, min(ps["num_classes"], pf["num_classes"]), (G,), generator=g) if pf["num_classes"] > 0 else None
    res = {}

    def gs(**kw):
        with contextlib.redirect_stdout(sys.stderr):
            return S.get_samples(early, postprocessing=S.predict_noise_postprocessing, num_channels=C, sample_height=H,
                                 sample_width=H, late_model=late, t_switch=T_SWITCH, device=dev, **kw)
    # (eta 0.1: sampler.py:116 takes sqrt(1 - abar_s - sigma_t^2), negative -> NaN for larger eta at 40 steps)
    ddim = dict(use_ddim=True, ddim_steps=40, ddim_eta=0.1)
    ddpm = dict(use_ddim=False, ddim_steps=50, ddim_eta=0.0)
    for label, nz, mode in (("ddim_injected_noise", noise, ddim), ("ddim_philox", None, ddim),
                            ("ddpm_1000_steps_philox", None, ddpm)):
        got = D.get_samples_sharded(gs, G, shape=(C, H, H), noise=nz, y=y, seed=11, **mode)
        if rank == 0:
            ref = gs(batch_size=G, seed=11, x_T=D.global_x_T(11, G, (C, H, H)), noise=nz,
                     y=y.to(dev) if y is not None else None, **mode)[0]
            assert np.isfinite(ref).all(), label
            res[label] = dict(equal=bool(np.array_equal(got.cpu().numpy(), ref)),
                              max_abs_diff=float(np.abs(got.cpu().numpy() - ref).max()), rows=G)
    # early exit: samples + both logs
    pe = CONFIGS["cifar10"]
    torch.manual_seed(4321)
    ee = ddb.EarlyExitUViT(ddb.UViT(**pe, max_batch=G), "mlp_probe_per_layer")
    synthetic_probes_(ee, pe["depth"], 1.0, 0.5)
    ee = ee.eval().to(dev)
    lo, hi = D.shard_bounds(G, rank, world)
    kw = dict(num_channels=3, sample_height=32, sample_width=32, threshold=0.08, depth=pe["depth"], device=dev)
    xT = D.global_x_T(5, G, (3, 32, 32))
    with contextlib.redirect_stdout(sys.stderr):
        s_loc, err_loc, idx_loc = ES.get_samples(ee, hi - lo, seed=5, x_T=xT[lo:hi], noise_row_offset=lo, **kw)
    s_all = D.all_gather_rows(torch.from_numpy(s_loc).to(dev), G)
    err_all, idx_all = D.gather_ee_logs(err_loc.to(dev), idx_loc.to(dev), G)
    if rank == 0:
        with contextlib.redirect_stdout(sys.stderr):
            s_ref, err_ref, idx_ref = ES.get_samples(ee, G, seed=5, x_T=xT, **kw)
        res["early_exit"] = dict(samples_equal=bool(np.array_equal(s_all.cpu().numpy(), s_ref)),
                                 indices_equal=bool(torch.equal(idx_all.cpu(), idx_ref)),
                                 probe_log_max_abs_diff=float((err_all.cpu() - err_ref).abs().max()),
                                 mean_exit_layer=float(idx_ref.mean()), rows=G)
        ok = (all(v["equal"] for k, v in res.items() if k != "early_exit") and res["early_exit"]["samples_equal"]
              and res["early_exit"]["indices_equal"] and res["early_exit"]["probe_log_max_abs_diff"] < 1e-5)
        print(json.dumps(dict(verify_shards=res, n_gpus=world, backend="nccl" if world > 1 else "none",
                              config=args.config, ok=ok)), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and not ok:
        raise SystemExit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=list(PAIRS), default="celeba")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: the config's BASELINE batch)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline sample")
    ap.add_argument("--decode", action="store_true",
                    help="latent configs: decode the samples with the KL autoencoder inside the timed regions")
    ap.add_argument("--ee", action="store_true", help="BASELINE config 3: early-exit sampling with exit compaction")
    ap.add_argument("--threshold", type=float, default=0.08)
    ap.add_argument("--slope", type=float, default=1.0, help="--ee: synthetic probe bias slope (sets the mean exit layer)")
    ap.add_argument("--wscale", type=float, default=0.5, help="--ee: synthetic probe weight scale (per-sample spread)")
    ap.add_argument("--full-run", action="store_true",
                    help="--impl reference: run the unmodified get_samples for all 1000 steps (config 1: --config cifar10 --batch 8)")
    ap.add_argument("--verify-shards", action="store_true", help="N-rank sharded == single-GPU, row for row (not a benchmark)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, <= 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl == "reference" or args.verify_shards):
        ap.error("--dump-outputs records the GPU sampling path: not with --impl reference or --verify-shards")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""  # the CPU arm: the reference's get_device() must pick the host
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # plain `python bench.py --gpus N`: re-launch under torchrun, one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"), __file__,
               *sys.argv[1:]]
        sys.exit(subprocess.call(cmd))
    if args.verify_shards:
        run_verify(args, rank, world, local_rank)
    elif args.ee:
        run_ee(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
