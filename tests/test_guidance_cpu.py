"""CPU tests of classifier-free guidance: the guided oracle (oracle/guidance_oracle.py) against the pinned unguided
oracle on the TINY_CLS spec, the `--cfg_scale` flag, the argument checks of get_samples, and the C-ABI symbol."""
import math

import pytest
import torch

from duodiff_b200 import _lib, sampler
from duodiff_b200.configs import CONFIGS
from oracle import guidance_oracle as G
from oracle import uvit_oracle as O
from tests.helpers import load_fixture, rel_l2, split_fixture

torch.set_num_threads(4)


@pytest.fixture(scope="module")
def tiny_cls():
    """The class-conditional TINY_CLS weights of tests/golden/make_golden.py (10 classes, [4, 8, 8] samples)."""
    sd, params = split_fixture(load_fixture("uvit_forward_tiny_cls"))
    spec = O.UViTSpec.from_params(params)
    return (lambda x, t, y: O.uvit_forward(sd, spec, x, t, y)), spec


def _inputs(spec, B=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    shape = (B, spec.in_chans, spec.img_size, spec.img_size)
    return torch.randn(shape, generator=g), torch.randn(1000, *shape, generator=g), \
        torch.randint(0, spec.num_classes - 1, (B,), generator=g)


def test_guided_oracle_at_scale_zero_is_the_unguided_sampler(tiny_cls):
    f, spec = tiny_cls
    x_T, noise, y = _inputs(spec)
    # a batch of 2B rows and one of B rows need not round alike: equal to fp32 summation-order noise
    ref = O.sample_ddpm(f, f, 950, x_T.clone(), noise, y=y, t_first=999, t_last=900)
    got = G.sample_ddpm_guided(f, f, 950, x_T.clone(), noise, y, 0.0, spec.num_classes - 1, t_first=999, t_last=900)
    assert rel_l2(got, ref) <= 1e-5
    ref = O.sample_ddim(f, None, float("inf"), x_T.clone(), noise, 20, 0.05, y=y)
    got = G.sample_ddim_guided(f, None, float("inf"), x_T.clone(), noise, 20, 0.05, y, 0.0, spec.num_classes - 1)
    assert rel_l2(got, ref) <= 1e-5


@pytest.mark.parametrize("rule", ["predict_noise", "predict_original"])
def test_guided_eps_is_the_composition_of_two_forwards(tiny_cls, rule):
    f, spec = tiny_cls
    x_T, noise, y = _inputs(spec, seed=1)
    null, s = spec.num_classes - 1, 1.5
    trace = {}
    G.sample_ddpm_guided(f, f, 995, x_T.clone(), noise, y, s, null, rule=rule, t_first=999, t_last=990, trace=trace)
    for k, t in enumerate(range(999, 989, -1)):
        x, tt = trace["x_in"][k], torch.full((x_T.shape[0],), float(t))
        c, u = f(x, tt, y), f(x, tt, torch.full_like(y, null))
        want = c + s * (c - u)
        assert rel_l2(trace["eps"][k], want) <= 1e-5, t
        assert rel_l2(want, c) > 1e-3, t  # guidance changed eps: the check is not vacuous


def test_combine_rounds_each_operation():
    c = torch.tensor([1.0, -2.5, 3.0e-8])
    u = torch.tensor([0.75, 1.0, -1.0e-8])
    d = (c - u)
    assert torch.equal(G.combine(c, u, 0.4), c + (0.4 * d))


def _base_argv():
    return ["--checkpoint_path", "a.pth", "--batch_size", "4", "--parametrization", "predict_noise",
            "--output_folder", "o", "--config_path", "c.yaml"]


def test_cfg_scale_flag():
    a = sampler.get_args(_base_argv())
    assert "cfg_scale" not in vars(a)  # unset: the namespace of the reference's flags, nothing more
    assert sorted(vars(a)) == sorted(["seed", "checkpoint_path", "checkpoint_path_late", "batch_size",
                                      "parametrization", "output_folder", "config_path", "config_path_late",
                                      "t_switch", "class_id", "use_ddim", "ddim_steps", "ddim_eta", "timesteps_save"])
    with pytest.raises(SystemExit):
        sampler.get_args(_base_argv() + ["--cfg_scale", "0.4"])
    a = sampler.get_args(_base_argv() + ["--class_id", "1", "--cfg_scale", "0.4"])
    assert a.cfg_scale == 0.4 and a.class_id == 1


def _small(name, **kw):
    import duodiff_b200 as ddb
    return ddb.UViT(**dict(CONFIGS[name], embed_dim=64, num_heads=2, depth=1, **kw))


def test_get_samples_rejects_bad_guidance():
    import duodiff_b200 as ddb
    kw = dict(batch_size=2, postprocessing=sampler.predict_noise_postprocessing, seed=0, num_channels=4,
              sample_height=32, sample_width=32)
    cond, y = _small("imagenet256_3"), torch.tensor([3, 4])
    with pytest.raises(ValueError, match="needs class labels"):
        sampler.get_samples(cond, cfg_scale=1.0, **kw)
    with pytest.raises(ValueError, match="class-conditional"):
        sampler.get_samples(_small("cifar10_3"), y=y, cfg_scale=1.0, **kw)
    with pytest.raises(ValueError, match="early exit"):
        sampler.get_samples(ddb.EarlyExitUViT(cond, "mlp_probe_per_layer"), y=y, cfg_scale=1.0, **kw)
    with pytest.raises(ValueError, match="outside"):
        sampler.get_samples(cond, y=y, cfg_scale=1.0, null_label=1001, **kw)
    with pytest.raises(ValueError, match="outside"):
        sampler.get_samples(cond, y=y, cfg_scale=1.0, late_model=_small("imagenet64_3"), null_label=1000, **kw)
    for bad in (math.nan, math.inf):
        with pytest.raises(ValueError, match="finite"):
            sampler.get_samples(cond, y=y, cfg_scale=bad, **kw)
    assert sampler._guidance([cond], y, 2, None) == (2.0, 1000)  # U-ViT's null row: the last of 1001


def test_guidance_symbol_is_exported():
    from duodiff_b200 import _build
    _build.build()
    assert "ddb_sampler_set_guidance" in _lib.EXPORTED_SYMBOLS
    assert hasattr(_lib.load(), "ddb_sampler_set_guidance")
