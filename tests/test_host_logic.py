"""CPU tests of the host-side logic: schedule/coefficients, hand-off rule, CLI surface, state_dict layout,
and that the C-ABI library loads and exports every symbol include/duodiff_b200.h declares."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from duodiff_b200 import _lib, ddpm, eesampler, sampler
from duodiff_b200.configs import CONFIGS
from tests.helpers import load_fixture

ROOT = Path(__file__).resolve().parents[1]


def test_library_exports_every_declared_symbol():
    from duodiff_b200 import _build
    _build.build()
    lib = _lib.load()
    header = (ROOT / "include" / "duodiff_b200.h").read_text()
    declared = set(re.findall(r"\b(ddb_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert set(_lib.EXPORTED_SYMBOLS) == declared
    assert b"sm_100a" in lib.ddb_version()


def test_no_gpu_means_loud_failure():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import duodiff_b200 as ddb
    net = ddb.UViT(**CONFIGS["celeba_3"])
    with pytest.raises(Exception):
        net(torch.zeros(1, 3, 64, 64), torch.zeros(1))


def test_schedule_matches_reference_bits():
    fx = load_fixture("schedule")
    s = ddpm.schedule()
    for k in fx:
        assert np.array_equal(s[k].numpy(), fx[k]), k


def test_step_coefficients():
    s = ddpm.schedule()
    tab, mode = ddpm.step_coefficients("predict_noise")
    assert mode == 0 and tab.shape == (1000, 4) and tab.dtype == torch.float32
    assert torch.equal(tab[:, 0], torch.sqrt(1 / s["alphas"]))
    assert torch.equal(tab[:, 1], (1 - s["alphas"]) / torch.sqrt(1 - s["alphas_bar"]))
    assert torch.equal(tab[:, 2], torch.sqrt(s["betas_tilde"])) and tab[0, 2] == 0  # beta_tilde_0 = 0 (Q4)
    tab_b, _ = ddpm.step_coefficients("predict_noise", variance="beta")  # ddpm_core.NoiseScheduler default
    assert torch.equal(tab_b[:, 2], torch.sqrt(s["betas"]))
    tab_p, mode_p = ddpm.step_coefficients("predict_previous")
    assert mode_p == 1 and tab_p[:, 0].eq(0).all() and tab_p[:, 1].eq(1).all()
    with pytest.raises(ValueError):
        ddpm.step_coefficients("predict_velocity")


@pytest.mark.parametrize("t_switch,expect", [(300, 700), (1, 999), (1000, 0), (0, -1), (1001, -1),
                                             (float("inf"), -1), (np.inf, -1), (300.5, -1), (-5, -1)])
def test_switch_step_follows_reference_quirks(t_switch, expect):
    """sampler.py:135-136: swap after the step at t == 1000 - t_switch (Q1); never for t_switch outside 1..1000."""
    assert ddpm.switch_step(t_switch) == expect
    # brute-force the reference loop
    model, used_late = "early", []
    for t in range(999, -1, -1):
        used_late.append(model == "late")
        if t == 1000 - t_switch:
            model = "late"
    first_late = next((999 - i for i, u in enumerate(used_late) if u), None)
    assert (first_late is None and expect <= 0) or first_late == expect - 1


def test_sampler_cli_flags_match_reference():
    a = sampler.get_args(["--checkpoint_path", "a.pth", "--batch_size", "4", "--parametrization", "predict_noise",
                          "--output_folder", "o", "--config_path", "c.yaml"])
    assert a.seed == 0 and a.t_switch == np.inf and a.checkpoint_path_late is None and a.timesteps_save == []
    assert a.use_ddim is False and a.ddim_steps == 50 and a.ddim_eta == 0.0 and a.class_id is None
    a = sampler.get_args(["--checkpoint_path", "a", "--checkpoint_path_late", "b", "--config_path", "c",
                          "--config_path_late", "d", "--t_switch", "300", "--batch_size", "128", "--parametrization",
                          "predict_original", "--output_folder", "o", "--timesteps_save", "1", "500", "--seed", "3"])
    assert a.t_switch == 300 and a.timesteps_save == [1, 500] and a.seed == 3
    with pytest.raises(SystemExit):
        sampler.get_args(["--parametrization", "nope"])
    e = eesampler.get_args(["--threshold", "0.08", "--checkpoint_path", "a", "--batch_size", "2", "--output_folder",
                            "o", "--config_path", "c"])
    assert e.threshold == 0.08 and e.seed == 0 and e.class_id is None


def test_rule_lookup_accepts_reference_function_objects():
    def predict_noise_postprocessing(model_output, x, t):  # same name as sampler.py:47
        raise AssertionError("never called")
    assert sampler._rule_name(predict_noise_postprocessing) == "predict_noise"
    assert sampler._rule_name(sampler.predict_original_postprocessing) == "predict_original"
    assert sampler._rule_name("predict_previous") == "predict_previous"
    with pytest.raises(ValueError):
        sampler._rule_name(lambda a, b, c: a)


def test_state_dict_layout_matches_reference_checkpoints():
    """Key order, names and shapes of SURVEY.md Q16, checked against the key list of a reference-generated fixture."""
    import duodiff_b200 as ddb
    fx = load_fixture("uvit_forward_tiny_cls")
    ref_keys = [k[3:] for k in fx if k.startswith("w::")]
    params = {k[3:]: v.item() for k, v in fx.items() if k.startswith("p::")}
    params["embed_dim"], params["num_heads"] = 32, 2
    net = ddb.UViT(**params)
    sd = net.state_dict()
    assert list(sd.keys()) == ref_keys
    assert all(tuple(sd[k].shape) == fx["w::" + k].shape for k in ref_keys)
    net.load_state_dict({k: torch.from_numpy(fx["w::" + k]) for k in ref_keys})  # loads a reference checkpoint
    fx = load_fixture("ee_forward_tiny")
    ref_keys = [k[3:] for k in fx if k.startswith("w::")]
    params = {k[3:]: v.item() for k, v in fx.items() if k.startswith("p::")}
    ee = ddb.EarlyExitUViT(ddb.UViT(**params), "mlp_probe_per_layer")
    assert list(ee.state_dict().keys()) == ref_keys
    assert len([k for k in ref_keys if k.startswith("uvit.")]) == len(ddb.UViT(**params).state_dict())
    d13 = ddb.UViT(**CONFIGS["celeba"])
    assert len(d13.state_dict()) == 164  # SURVEY.md Q16
    assert len(ddb.EarlyExitUViT(d13, "mlp_probe_per_layer").state_dict()) == 268
    # the timestep-indexed MLP probe layouts carry the reference's ModuleDict keys (models/early_exit.py:228-239)
    d3 = ddb.UViT(**CONFIGS["celeba_3"])
    pt = ddb.EarlyExitUViT(d3, "mlp_probe_per_timestep").state_dict()
    assert "matrix.999.classifier.0.weight" in pt and sum(k.startswith("matrix.") for k in pt) == 2000
    from duodiff_b200.early_exit import probe_keys
    keys = probe_keys("mlp_probe_per_layer_per_timestep", 3)
    assert keys[:4] == ["0, 0", "1, 0", "2, 0", "0, 1"] and len(keys) == 3000
    ap = ddb.EarlyExitUViT(d3, "attention_probe").state_dict()  # the reference's default classifier_type
    fa = load_fixture("ee_attention_probe_tiny")
    ref_keys = {k[len("u::w::"):] for k in fa if k.startswith("u::w::matrix.0.")}
    assert ref_keys == {k for k in ap if k.startswith("matrix.0.")} and len(ref_keys) == 7
    assert tuple(ap["matrix.0.q"].shape) == (1, 1, 1, 512) and tuple(ap["matrix.2.weight_kv.weight"].shape) == (1024, 512)
    fx = load_fixture("ee_probe_types_tiny")  # key spelling as saved by the reference's own state_dict()
    assert "plt::w::matrix.2, 321.classifier.0.bias" in fx and "pt::w::matrix.7.classifier.0.weight" in fx


def test_constructor_variants_have_the_reference_parameter_tree():
    """mlp_time_embed / conv / skip / qk_scale / use_checkpoint of models/uvit.py:229-247: same state_dict keys and shapes
    as the reference's own modules (fixture written from their state_dict())."""
    import duodiff_b200 as ddb
    fx = load_fixture("uvit_variants_tiny")
    for tag in ("a", "b"):
        ref = {k[len(f"{tag}::w::"):]: v.shape for k, v in fx.items() if k.startswith(f"{tag}::w::")}
        params = {k[len(f"{tag}::p::"):]: v.item() for k, v in fx.items() if k.startswith(f"{tag}::p::")}
        own = {k: tuple(v.shape) for k, v in ddb.UViT(**params, use_checkpoint=True).state_dict().items()}
        assert own == {k: tuple(s) for k, s in ref.items()}, tag
    assert "final_layer.weight" not in ddb.UViT(**dict(CONFIGS["celeba_3"], conv=False)).state_dict()
    head = ddb.OutputHead(512, 48, 3, conv=False)
    assert isinstance(head.final_layer, torch.nn.Identity)


def test_unsupported_options_raise():
    import duodiff_b200 as ddb
    with pytest.raises(NotImplementedError):
        ddb.UViT(**CONFIGS["celeba_3"], norm_layer=torch.nn.BatchNorm1d)
    with pytest.raises(ValueError):
        ddb.EarlyExitUViT(ddb.UViT(**CONFIGS["celeba_3"]), "linear_probe")
    with pytest.raises(NotImplementedError):
        ddb.AttentionProbe(512, num_heads=2)


def test_config_filter_drops_stray_keys(tmp_path):
    from duodiff_b200 import _io
    (tmp_path / "c.yaml").write_text("model_params:\n  img_size: 64\n  patch_size: 4\n  in_chans: 3\n  embed_dim: 768\n"
                                     "  depth: 17\n  num_heads: 12\n  mlp_ratio: 4\n  qkv_bias: False\n"
                                     "  mlp_time_embed: False\n  num_classes: 1000\n  normalize_timesteps: False\n"
                                     "  classifier_type: \"mlp_per_layer\"\n")
    kw = _io.uvit_kwargs(_io.load_config(tmp_path / "c.yaml"))
    assert "classifier_type" not in kw and kw["depth"] == 17  # Q14: the reference raises TypeError here
    with pytest.raises(FileNotFoundError):
        _io.load_config(tmp_path / "missing.yaml")


def test_bench_flop_model_matches_survey():
    import bench
    f3, f13 = bench.forward_flops(CONFIGS["celeba_3"]), bench.forward_flops(CONFIGS["celeba"])
    assert abs(f3["total"] / 1e9 - 5.552) < 0.01 and abs(f13["total"] / 1e9 - 24.421) < 0.01  # SURVEY.md §8d
    f = bench.forward_flops(CONFIGS["imagenet256"])
    assert abs(f["total"] / 1e9 - 152.912) < 0.05


def test_ddim_plan_matches_reference_call_pattern():
    """Host-side DDIM plan (timesteps + which backbone) against the hooks recorded on the unmodified reference
    (tests/golden/ddim_sampler_tiny.npz): strided schedule and the `t < 1000 - t_switch` hand-off after the step."""
    from duodiff_b200.ddpm import ddim_coefficients, ddim_timesteps
    from duodiff_b200.sampler import _ddim_plan
    from tests.helpers import load_fixture
    fx = load_fixture("ddim_sampler_tiny")
    for steps, eta in ((50, 0.0), (20, 0.05)):
        key = f"{steps}_{eta}"
        ts, flags = _ddim_plan(steps, True, 300)
        assert [t for t, f in zip(ts, flags) if not f] == fx[f"early_ts_{key}"].tolist()
        assert [t for t, f in zip(ts, flags) if f] == fx[f"late_ts_{key}"].tolist()
        table, mode = ddim_coefficients(steps, eta)
        assert mode == 2 and table.shape == (1000, 4)
        last_t = ddim_timesteps(steps)[-2]
        assert table[last_t, 2].item() == 0.0  # z = 0 for the last pair (s == 0)
        assert (table[[t for t in range(1000) if t not in ts]] == 0).all()
    ts, flags = _ddim_plan(50, False, 300)
    assert not any(flags)
    with pytest.raises(ValueError):
        ddim_timesteps(2000)


def test_autoencoder_shim_surface():
    """duodiff_b200.autoencoder mirrors models/utils/autoencoder.py:452-516 for the decode side: same constructor
    arguments and default ddconfig; unsupported decoder options raise; no CUDA device -> loud error, no fallback."""
    from duodiff_b200 import _lib
    from duodiff_b200.autoencoder import DEFAULT_DDCONFIG, FrozenAutoencoderKL, get_autoencoder
    assert DEFAULT_DDCONFIG["ch_mult"] == [1, 2, 4, 4] and DEFAULT_DDCONFIG["resolution"] == 256
    for bad in (dict(attn_resolutions=[16]), dict(use_linear_attn=True), dict(tanh_out=True)):
        with pytest.raises(NotImplementedError):
            FrozenAutoencoderKL(dict(DEFAULT_DDCONFIG, **bad), 4, state_dict={})
    with pytest.raises(ValueError):
        FrozenAutoencoderKL(DEFAULT_DDCONFIG, 4)
    if not torch.cuda.is_available():
        with pytest.raises(_lib.DuoDiffError, match="no CPU fallback"):
            FrozenAutoencoderKL(DEFAULT_DDCONFIG, 4, state_dict={})
    with pytest.raises(FileNotFoundError):
        get_autoencoder("/nonexistent/autoencoder_kl.pth")
    assert _lib.AEConfig.ch_mult.size == 32  # int32[8], include/duodiff_b200.h


def test_output_side_files(tmp_path):
    """sampler.py:158-189 / eesampler.py:92-111: file names, the sqrt-grid, clipping, statistics.txt and the .pt logs.
    Pixel values follow plt.imsave (x * 255 truncated to uint8, opaque alpha)."""
    from PIL import Image
    from duodiff_b200 import eesampler, sampler
    rng = np.random.default_rng(0)
    samples = rng.uniform(-0.2, 1.2, size=(5, 8, 8, 3)).astype(np.float32)
    sampler.dump_samples(samples, tmp_path)
    sampler.dump_samples(samples[:2], tmp_path, 250)
    sampler.dump_statistics(1.5, tmp_path)
    names = sorted(p.name for p in tmp_path.iterdir())
    assert names == sorted([f"{i}.png" for i in range(5)] + ["0_250.png", "1_250.png", "grid_image.png",
                                                             "statistics.txt"])
    img = np.asarray(Image.open(tmp_path / "3.png"))
    assert img.shape == (8, 8, 4) and (img[..., 3] == 255).all()
    assert np.array_equal(img[..., :3], (np.clip(samples[3], 0, 1) * 255).astype(np.uint8))
    grid = np.asarray(Image.open(tmp_path / "grid_image.png"))
    assert grid.shape == (16, 16, 4)  # the second call (2 samples -> ceil(sqrt(2)) = 2) overwrote the 3x3 grid
    assert (tmp_path / "statistics.txt").read_text() == "Elapsed time: 1.5 s\n"
    out = tmp_path / "ee"
    out.mkdir()
    eesampler.dump_samples(samples, out)
    eesampler.dump_statistics(2.0, torch.zeros(1000, 3), torch.ones(1000, 5), out)
    assert sorted(p.name for p in out.iterdir()) == sorted(
        [f"{i}.png" for i in range(5)] + ["statistics.txt", "error_prediction_by_timestep.pt",
                                          "indices_by_timestep.pt"])
    assert torch.load(out / "indices_by_timestep.pt").shape == (1000, 5)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours): one JSON line with the contract's keys,
    the GPU arm's metric / unit / config, e2e == value with zero copy bytes, a cpu_baseline describing the sample."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parents[1]
    res = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/sec" and d["higher_is_better"] is True
    assert d["metric"].startswith("images/sec (DuoDiff sampling") and "celeba" in d["config"]["workload"]
    assert d["config"]["batch_per_gpu"] == 128 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["e2e"] == dict(value=d["value"], unit="images/sec", h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["value"] > 0 and d["gpu_launches"] == 0


def test_bench_dump_outputs_fit_the_limit_and_repeat(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float32 .npy files within DUMP_LIMIT bytes in all; an array that fits is written
    whole, a larger one as the same seeded sample of its rows on every call."""
    import importlib.util
    import subprocess
    import sys
    spec = importlib.util.spec_from_file_location("_bench", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "DUMP_LIMIT", 1 << 20)
    g = torch.Generator().manual_seed(0)
    samples = torch.rand(80, 32, 32, 3, generator=g)  # 960 KB
    exit_log = torch.randint(0, 13, (1000, 80), generator=g, dtype=torch.int32)  # 312 KB
    bench.dump_outputs(str(tmp_path), dict(samples=samples, exit_log=exit_log))
    files = sorted(tmp_path.iterdir())
    assert [p.name for p in files] == ["exit_log.npy", "samples.npy"]
    assert sum(p.stat().st_size for p in files) <= 1 << 20
    log, got = np.load(tmp_path / "exit_log.npy"), np.load(tmp_path / "samples.npy")
    assert log.dtype == got.dtype == np.float32 and np.array_equal(log, exit_log.numpy())
    assert 0 < len(got) < 80 and got.shape[1:] == (32, 32, 3)
    rows = [i for r in got for i in range(80) if np.array_equal(r, samples[i].numpy())]
    assert rows == sorted(set(rows)) and len(rows) == len(got)  # distinct rows of the output, in order
    bench.dump_outputs(str(tmp_path), dict(samples=samples, exit_log=exit_log))
    assert np.array_equal(np.load(tmp_path / "samples.npy"), got)
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert res.returncode == 2 and "--steps" in res.stderr


def test_cli_labels_follow_the_reference_draw_modulo_num_classes():
    """sampler.py:314-318: `--class_id` draws torch.randint(1, 1001, (B,)) after seed_everything(seed).  The shims keep
    that draw and take it modulo num_classes (documented deviation: label 1000 cannot index a 1000-row table)."""
    torch.manual_seed(11)
    ref = torch.randint(1, 1001, (4096,))
    torch.manual_seed(11)
    y = sampler.draw_labels(4096, 1000)
    assert y.dtype == torch.int64 and int(y.min()) >= 0 and int(y.max()) <= 999
    ok = ref < 1000
    assert torch.equal(y[ok], ref[ok]) and y[~ok].eq(0).all()  # only the reference's out-of-range label changes
    torch.manual_seed(11)
    assert torch.equal(sampler.draw_labels(4096, 1001), ref)  # ImageNet-256 configs: 1001 classes, nothing changes
    assert eesampler.draw_labels is sampler.draw_labels


def test_top_level_cli_shims_reexport_the_reference_names():
    """`python sampler.py ...` / `python eesampler.py ...` work from the repository root like in the reference."""
    import importlib.util
    for name, mod, names in (("sampler.py", sampler, ("main", "get_samples", "get_args", "dump_samples",
                                                      "dump_statistics", "predict_noise_postprocessing",
                                                      "predict_original_postprocessing",
                                                      "predict_previous_postprocessing")),
                             ("eesampler.py", eesampler, ("main", "get_samples", "get_args", "dump_samples",
                                                          "dump_statistics"))):
        spec = importlib.util.spec_from_file_location("_shim_" + name[:-3], ROOT / name)
        shim = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(shim)
        for n in names:
            assert getattr(shim, n) is getattr(mod, n), (name, n)


def test_engine_rejects_threshold_free_early_exit_flag_confusion():
    """Early exit is switched by ee_mode, not by the sign of the threshold (ADVICE r1): the Sampler passes ee_mode = -1
    exactly when no threshold is given."""
    import inspect
    src = inspect.getsource(ddpm.Sampler.__init__)
    assert "-1 if ee_threshold is None" in src


def test_fid_shim_reads_cli_outputs_and_frechet_closed_form(tmp_path):
    """fid.py keeps the reference's command line (fid.py:8-31) and sample reader (utils/evaluation_utils.py:13-24); the
    metric itself needs torchmetrics + pretrained InceptionV3 (not bundled) and must say so."""
    import importlib.util
    from duodiff_b200 import _io
    spec = importlib.util.spec_from_file_location("_shim_fid", ROOT / "fid.py")
    fid = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fid)
    rng = np.random.default_rng(0)
    samples = rng.random((5, 8, 8, 3)).astype(np.float32)
    _io.dump_samples(samples, tmp_path)  # what sampler.py writes: 0.png .. 4.png + grid_image.png
    got = fid.read_samples(tmp_path)
    assert got.shape == (5, 3, 8, 8) and got.dtype == torch.float32  # the grid image is skipped
    want = torch.from_numpy((samples * 255).astype(np.uint8).astype(np.float32) / 255).permute(0, 3, 1, 2)
    assert torch.equal(got, want)
    args = fid.get_args(["--dataset", "celeba", "--samples_path", str(tmp_path)])
    assert args.seed == 0 and args.data_path == "data"
    # Frechet distance: identical Gaussians -> 0; diagonal case has the closed form sum (sqrt(a) - sqrt(b))^2 + |dmu|^2
    a, b = rng.random(6) + 0.5, rng.random(6) + 0.5
    mu = rng.random(6)
    assert abs(fid.frechet_distance(mu, np.diag(a), mu, np.diag(a))) < 1e-9
    want = ((np.sqrt(a) - np.sqrt(b)) ** 2).sum() + 0.25 * 6
    assert abs(fid.frechet_distance(mu, np.diag(a), mu + 0.5, np.diag(b)) - want) < 1e-9
    try:
        import torchmetrics  # noqa: F401
    except ImportError:
        with pytest.raises(RuntimeError, match="torchmetrics"):
            fid.fid_evaluation(got, got)
