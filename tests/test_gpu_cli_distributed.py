"""GPU tests of the two command lines under torchrun: `python -m torch.distributed.run --standalone --nproc-per-node 2
sampler.py …` writes the same files as a plain `python sampler.py …` with the same arguments -- byte for byte,
except statistics.txt (a time) and eesampler's batch-mean probe log (a weighted mean of the shards' means).  Both
ranks share one GPU (gloo allows that); with two or more GPUs one case also runs with a GPU per rank."""
import os
import sys
from pathlib import Path

import pytest
import torch
import yaml

from tests.helpers import CONFIGS
from tests.process_tree import run_tree
from tests.test_gpu_cli import _write

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
TIMEOUT = 900


def _first_gpu_only():
    """Environment in which both ranks see the same single GPU."""
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    return dict(os.environ, CUDA_VISIBLE_DEVICES=visible.split(",")[0] if visible else "0")


def _run(cmd, env=None):
    """Run `cmd` from the repository root; on timeout no rank outlives the test (tests/process_tree.py)."""
    rc, out = run_tree(cmd, TIMEOUT, cwd=ROOT, env=env)
    if rc is None:
        pytest.fail(f"timed out after {TIMEOUT} s: {' '.join(cmd)}\n{out[-4000:]}")
    if rc != 0:
        pytest.fail(f"exit code {rc}: {' '.join(cmd)}\n{out[-4000:]}")
    return out


def _compare(script, args, tmp: Path, env=None, nproc=2):
    """Run `script` once plainly and once under torchrun with `nproc` ranks; return the two output folders after
    checking that they hold the same files and that every file but statistics.txt and the probe log is identical."""
    single, multi = tmp / "single", tmp / f"torchrun{nproc}"
    _run([sys.executable, script, *args, "--output_folder", str(single)], env=env)
    out = _run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(nproc), script,
                *args, "--output_folder", str(multi)], env=env)
    assert "Gathered" in out and "Using device" in out
    names = sorted(p.name for p in single.iterdir())
    assert names == sorted(p.name for p in multi.iterdir())
    assert (multi / "statistics.txt").read_text().startswith("Elapsed time: ")
    for name in names:
        if name in ("statistics.txt", "error_prediction_by_timestep.pt"):
            continue
        if name.endswith(".pt"):
            assert torch.equal(torch.load(single / name), torch.load(multi / name)), name
        else:
            assert (single / name).read_bytes() == (multi / name).read_bytes(), name
    return single, multi, names


def _duodiff_args(tmp):
    ck_e, cfg_e = _write(tmp, "early", CONFIGS["cifar10_3"], 1, wrap=False)
    ck_l, cfg_l = _write(tmp, "late", CONFIGS["cifar10"], 2, wrap=True)
    return ["--checkpoint_path", ck_e, "--config_path", cfg_e, "--checkpoint_path_late", ck_l, "--config_path_late",
            cfg_l, "--t_switch", "300", "--batch_size", "5", "--parametrization", "predict_noise", "--seed", "3",
            "--timesteps_save", "500", "900"]


def test_torchrun_duodiff_ddpm_uneven_shards(tmp_path):
    """DuoDiff pair, 5 images over 2 ranks (3 + 2), intermediates at t = 500 and 900."""
    _, _, names = _compare("sampler.py", _duodiff_args(tmp_path), tmp_path, env=_first_gpu_only())
    assert len(names) == 5 + 1 + 1 + 10  # samples, grid, statistics, intermediates


def test_torchrun_duodiff_one_gpu_per_rank(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: this machine has one, and the shared-GPU case runs above")
    _compare("sampler.py", _duodiff_args(tmp_path), tmp_path)


def test_torchrun_ddim_class_conditional(tmp_path):
    ck, cfg = _write(tmp_path, "in64", CONFIGS["imagenet64_3"], 5, wrap=True, extra={"classifier_type": "attention_probe"})
    args = ["--checkpoint_path", ck, "--config_path", cfg, "--batch_size", "3", "--parametrization", "predict_noise",
            "--use_ddim", "--ddim_steps", "20", "--ddim_eta", "0.02", "--class_id", "7", "--seed", "1"]
    _compare("sampler.py", args, tmp_path, env=_first_gpu_only())


def test_torchrun_latent_decode_with_an_empty_shard(tmp_path):
    """One image over 2 ranks: rank 1 builds nothing and still joins the gather of the decoded 256x256 images."""
    from oracle.ae_oracle import AESpec, random_state_dict
    ae = tmp_path / "ae.pth"
    torch.save(random_state_dict(AESpec(), 9), ae)
    ck, cfg = _write(tmp_path, "in256", CONFIGS["imagenet256_3"], 10, wrap=False)
    c = yaml.safe_load(Path(cfg).read_text())
    c["autoencoder"] = {"autoencoder_checkpoint_path": str(ae)}
    Path(cfg).write_text(yaml.safe_dump(c))
    args = ["--checkpoint_path", ck, "--config_path", cfg, "--batch_size", "1", "--parametrization", "predict_noise",
            "--use_ddim", "--ddim_steps", "10", "--class_id", "1", "--seed", "4"]
    _, multi, names = _compare("sampler.py", args, tmp_path, env=_first_gpu_only())
    assert names == ["0.png", "grid_image.png", "statistics.txt"]
    from PIL import Image
    assert Image.open(multi / "0.png").size == (256, 256)


def test_torchrun_eesampler(tmp_path):
    ck, cfg = _write(tmp_path, "ee", CONFIGS["cifar10"], 6, wrap=False, ee=True)
    args = ["--checkpoint_path", ck, "--config_path", cfg, "--threshold", "0.45", "--batch_size", "5", "--seed", "2"]
    single, multi, _ = _compare("eesampler.py", args, tmp_path, env=_first_gpu_only())
    e1 = torch.load(single / "error_prediction_by_timestep.pt")
    e2 = torch.load(multi / "error_prediction_by_timestep.pt")
    assert e1.shape == e2.shape == (1000, 13) and e1.dtype == e2.dtype
    assert torch.isfinite(e2).all() and float((e1 - e2).abs().max()) <= 1e-5
    idx = torch.load(multi / "indices_by_timestep.pt")
    assert idx.shape == (1000, 5) and float(idx.min()) < 13  # exits happened
