"""Host-side checks of the KL-autoencoder encode surface (no device needed): the oracle's encoder restatement, the
random-init encoder weights of duodiff_b200.autoencoder, and the stride-2 tap addressing the Downsample kernel uses."""
import pytest
import torch
import torch.nn.functional as F

from duodiff_b200 import _lib
from duodiff_b200.autoencoder import DEFAULT_DDCONFIG, FrozenAutoencoderKL, random_init_state_dict
from oracle import ae_encoder_oracle as E
from oracle import ae_oracle as A


def _full_sd(spec, seed):
    sd = A.random_state_dict(spec, seed)
    sd.update(E.random_encoder_state_dict(spec, seed + 1))
    return sd


def test_oracle_encode_moments_shapes_and_taps():
    spec = E.AEEncSpec(ch=32, ch_mult=[1, 2, 2], num_res_blocks=1, resolution=32)
    sd = E.random_encoder_state_dict(spec, 0)
    x = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(1))
    tap = {}
    m = E.encode_moments(sd, spec, x, tap)
    assert m.shape == (2, 2 * spec.embed_dim, spec.z_res, spec.z_res) and bool(torch.isfinite(m).all())
    assert torch.equal(tap["moments"], m)
    expect = {
        "conv_in": (32, 32, 32),
        "down.0.block.0.norm1": (32, 32, 32), "down.0.block.0.conv2+res": (32, 32, 32),
        "down.0.downsample": (32, 16, 16),
        "down.1.block.0.conv1": (64, 16, 16), "down.1.block.0.conv2+nin": (64, 16, 16),
        "down.1.downsample": (64, 8, 8),
        "down.2.block.0.conv2+res": (64, 8, 8),
        "mid.block_1.conv2+res": (64, 8, 8), "mid.attn_1.norm": (64, 8, 8), "mid.attn_1.pv": (64, 8, 8),
        "mid.attn_1.proj_out+res": (64, 8, 8), "mid.block_2.conv2+res": (64, 8, 8), "norm_out": (64, 8, 8),
    }
    for name, chw in expect.items():
        assert tuple(tap[name].shape) == (2, *chw), name
    assert "down.2.downsample" not in tap  # the last level keeps its resolution
    assert not any(k.startswith("up.") for k in tap)


def test_oracle_sample_formula():
    g = torch.Generator().manual_seed(2)
    mom = torch.randn(2, 8, 4, 4, generator=g) * 20  # logvar beyond both clamp bounds
    n = torch.randn(2, 4, 4, 4, generator=g)
    z = E.sample(mom, n, 0.5)
    mean, logvar = mom[:, :4], mom[:, 4:].clamp(-30, 20)
    assert torch.allclose(z, 0.5 * (mean + torch.exp(0.5 * logvar) * n))


def test_random_init_encoder_keys_match_oracle():
    full = random_init_state_dict(DEFAULT_DDCONFIG, 4, 0, encoder=True)
    dec = random_init_state_dict(DEFAULT_DDCONFIG, 4, 0)
    assert not any(k.startswith(("encoder.", "quant_conv.")) for k in dec)
    for k, v in dec.items():  # the default (decoder-only) output is unchanged by the encoder keys
        assert torch.equal(full[k], v), k
    enc = {k: tuple(v.shape) for k, v in full.items() if k not in dec}
    ref = {k: tuple(v.shape) for k, v in E.random_encoder_state_dict(E.AEEncSpec(), 0).items()}
    assert enc == ref
    assert ref["encoder.conv_in.weight"] == (128, 3, 3, 3) and ref["quant_conv.weight"] == (8, 8, 1, 1)
    assert ref["encoder.conv_out.weight"] == (8, 512, 3, 3)
    assert sum(k.endswith("downsample.conv.weight") for k in ref) == 3


def test_stride2_box_addressing_is_padded_stride2_conv():
    """The Downsample kernel reads tap (ky, kx) of output pixel (y, x) from the 5-D view {(q, c), x', p, y', b} of the
    source at (q, x', p, y') = (kx & 1, x + (kx >> 1), ky & 1, y + (ky >> 1)), zero past the right / bottom edge.
    Emulated here with the same coordinates: equals F.pad(h, (0, 1, 0, 1)) then a 3x3 stride-2 convolution."""
    g = torch.Generator().manual_seed(3)
    B, C, H, N = 2, 5, 8, 6
    h = torch.randn(B, C, H, H, generator=g, dtype=torch.float64)
    w = torch.randn(N, C, 3, 3, generator=g, dtype=torch.float64)
    ref = F.conv2d(F.pad(h, (0, 1, 0, 1)), w, stride=2)
    # 5-D view of the NHWC source: view[b, y', p, x', q, c] = h[b, c, 2y' + p, 2x' + q]
    view = h.permute(0, 2, 3, 1).reshape(B, H // 2, 2, H // 2, 2, C)
    Ho = H // 2
    out = torch.zeros(B, N, Ho, Ho, dtype=torch.float64)
    for ky in range(3):
        for kx in range(3):
            q, dx, p, dy = kx & 1, kx >> 1, ky & 1, ky >> 1
            box = torch.zeros(B, Ho, Ho, C, dtype=torch.float64)  # TMA zero fill outside the tensor
            box[:, :Ho - dy, :Ho - dx] = view[:, dy:, p, dx:, q]
            out += torch.einsum("byxc,nc->bnyx", box, w[:, :, ky, kx])
    assert torch.allclose(out, ref)


def test_python_surface_without_a_device():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    sd = _full_sd(E.AEEncSpec(ch=64, ch_mult=[1, 2], num_res_blocks=1, resolution=32), 0)
    dd = dict(DEFAULT_DDCONFIG, ch=64, ch_mult=[1, 2], num_res_blocks=1, resolution=32)
    with pytest.raises(_lib.DuoDiffError, match="no CPU fallback"):
        FrozenAutoencoderKL(dd, 4, state_dict=sd)
    for name in ("encode", "encode_moments", "sample", "forward"):
        assert callable(getattr(FrozenAutoencoderKL, name))
