"""GPU parity tests of the KL-autoencoder encode (run with `-m gpu` on a B200): Encoder + quant_conv + sample through the
C ABI (ddb_ae_create_encoder / ddb_ae_encode_moments / ddb_ae_sample) against oracle/ae_encoder_oracle.py (fp32).

Tolerances (NHWC bf16 activations between layers, bf16 tensor-core operands, fp32 accumulation and GroupNorm
statistics, quant_conv folded into conv_out's weights in fp32 before the bf16 rounding); the bounds are decode's
(tests/test_gpu_autoencoder.py), measured values on a B200 in brackets:
  * every tapped layer, free-running                       : rel-L2 <= 2.5e-2 [2.7e-3 .. 9.4e-3]
  * moments (mean | logvar)                                : rel-L2 <= 2e-2   [8.3e-3 .. 9.2e-3]
                                                             max-abs <= 3e-2 * max|ref|
  * sample with injected noise vs the oracle formula       : fp32 rounding (rtol 4e-6, atol 1e-6) [0]
  * chunked == unchunked, sample alone == sample in a batch : bit-exact (GroupNorm partials reduced in a fixed order)
"""
import pytest
import torch

from oracle import ae_encoder_oracle as E
from oracle import ae_oracle as A
from tests.helpers import rel_l2

pytestmark = pytest.mark.gpu

LAYER_REL_L2 = 2.5e-2
OUT_REL_L2 = 2e-2
OUT_MAX_ABS = 3e-2


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.set_num_threads(16)
    return torch.device("cuda:0")


def _dd(spec):
    return dict(double_z=True, z_channels=spec.z_channels, resolution=spec.resolution, in_channels=spec.in_channels,
                out_ch=spec.out_ch, ch=spec.ch, ch_mult=spec.ch_mult, num_res_blocks=spec.num_res_blocks,
                attn_resolutions=[], dropout=0.0)


def _sd(spec, seed, encoder=True):
    sd = A.random_state_dict(spec, seed)
    if encoder:
        sd.update(E.random_encoder_state_dict(spec, seed + 100))
    return sd


def _make(spec, seed, max_batch, encoder=True):
    from duodiff_b200.autoencoder import FrozenAutoencoderKL
    sd = _sd(spec, seed, encoder)
    ae = FrozenAutoencoderKL(_dd(spec), spec.embed_dim, state_dict=sd, scale_factor=spec.scale_factor,
                             max_batch=max_batch)
    return ae, sd


def _images(spec, B, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, spec.in_channels, spec.resolution, spec.resolution, generator=g) * 2 - 1


def _check_out(out, ref):
    e = rel_l2(out, ref)
    print(f"moments rel-L2 {e:.2e}")
    assert e <= OUT_REL_L2, e
    assert float((out - ref).abs().max()) <= OUT_MAX_ABS * float(ref.abs().max())


SMALL = E.AEEncSpec(ch=64, ch_mult=[1, 2], num_res_blocks=1, resolution=32)


@pytest.mark.parametrize("spec,B", [
    (SMALL, 2),                                                                 # downsample to a 16x16 grid
    (E.AEEncSpec(ch=64, ch_mult=[1, 2, 2], num_res_blocks=1, resolution=128), 3),  # two downsamples, 128-wide rows
])
def test_encode_layer_by_layer(dev, spec, B):
    """Every layer the encoder's launch list exposes (conv_in over the im2col rows, both convolutions and GroupNorms of
    every ResnetBlock incl. the nin_shortcut K-extension, the stride-2 Downsample convolutions, the AttnBlock,
    norm_out) against the oracle's taps, then the moments."""
    ae, sd = _make(spec, 3, B)
    x = _images(spec, B, 4)
    tap = {}
    ref = E.encode_moments(sd, spec, x, tap)
    xc = x.to(dev)
    seen = set()
    for i, (name, c, h, w, _f32) in enumerate(ae.encoder_ops()):
        if c == 0 or name not in tap:
            continue
        _m, dump = ae.encode_debug(xc, i)
        t = tap[name]
        assert dump.shape[1:] == t.shape[1:], name
        e = rel_l2(dump.cpu(), t)
        print(f"  {name:28s} rel-L2 {e:.2e}")
        assert e <= LAYER_REL_L2, (name, e)
        seen.add(name.rsplit(".", 1)[-1])
    assert {"conv_in", "norm1", "conv1", "norm2", "conv2+res", "conv2+nin", "downsample", "norm", "pv",
            "proj_out+res", "norm_out"} <= seen
    out = ae.encode_moments(xc)
    assert out.shape == ref.shape
    _check_out(out.cpu(), ref)


def test_default_config_matches_oracle_and_is_batch_invariant(dev):
    """get_autoencoder's ddconfig (3x256x256 -> 8x32x32 moments): B = 3 in chunks of 2 against the oracle (fp32 on the
    GPU, TF32 off); the level-0 Downsample (N = 128) runs the two-tile (MT = 2) path.  Chunking and batch position
    must not change a single bit."""
    spec = E.AEEncSpec()
    ae, sd = _make(spec, 7, 2)
    x = _images(spec, 3, 8)
    xc = x.to(dev)
    out = ae.encode_moments(xc)
    assert out.shape == (3, 8, 32, 32) and bool(torch.isfinite(out).all())
    sdc = {k: v.to(dev) for k, v in sd.items()}
    with torch.no_grad():
        ref = E.encode_moments(sdc, spec, xc[:2])
    _check_out(out[:2].cpu(), ref.cpu())
    alone = ae.encode_moments(xc[2:3])
    assert torch.equal(alone[0], out[2])
    swapped = ae.encode_moments(xc[[1, 0]])
    assert torch.equal(swapped[0], out[1]) and torch.equal(swapped[1], out[0])
    del ae
    whole, _ = _make(spec, 7, 3)  # one chunk of 3
    assert torch.equal(whole.encode_moments(xc), out)
    prof = whole.profile_encode(xc)
    assert abs(sum(v["flops"] for v in prof.values()) / 3 / 1e9 - 272.7) < 0.1  # algorithmic GFLOP / image
    assert all(v["ms"] >= 0 for v in prof.values())


def test_sample_and_forward(dev):
    ae, _sd = _make(SMALL, 5, 2)
    x = _images(SMALL, 2, 6).to(dev)
    m = ae.encode_moments(x)
    m[:, 4:, 0, 0] = torch.tensor([-40.0, 25.0], device=dev)[:, None]  # both clamp bounds
    noise = torch.randn(2, 4, 16, 16, device=dev)
    z = ae.sample(m, noise)
    ref = E.sample(m, noise, SMALL.scale_factor)
    print(f"sample max-abs diff {float((z - ref).abs().max()):.2e}")
    torch.testing.assert_close(z, ref, rtol=4e-6, atol=1e-6)

    torch.manual_seed(9)
    a = ae.encode(x)
    torch.manual_seed(9)
    b = ae.sample(ae.encode_moments(x))
    assert torch.equal(a, b) and a.shape == (2, 4, 16, 16)
    torch.manual_seed(9)
    assert torch.equal(ae(x, "encode"), a)
    assert torch.equal(ae.forward(x, "encode_moments"), ae.encode_moments(x))
    assert torch.equal(ae(a, "decode"), ae.decode(a))
    with pytest.raises(NotImplementedError):
        ae(x, "reconstruct")


def test_decode_untouched_by_the_encoder(dev):
    """decode(z) -> encode(x) -> decode(z) on one handle gives the same image bit for bit (the encoder reuses the
    decoder's workspace), the decoder's launch list is unchanged, and a decode-only state_dict still decodes."""
    from duodiff_b200._lib import DuoDiffError
    ae, _sd = _make(SMALL, 11, 2)
    z = torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(12)).to(dev) * SMALL.scale_factor
    ops0 = ae.ops()
    img0 = ae.decode(z)
    ae.encode(_images(SMALL, 2, 13).to(dev))
    assert torch.equal(ae.decode(z), img0)
    assert ae.ops() == ops0

    dec_only, sd = _make(SMALL, 11, 2, encoder=False)
    assert torch.equal(dec_only.decode(z), img0)
    with pytest.raises(DuoDiffError, match="missing"):
        dec_only.encode(_images(SMALL, 1, 0).to(dev))
    with pytest.raises(DuoDiffError, match="missing"):  # and again: no half-built encoder is left behind
        dec_only.encode_moments(_images(SMALL, 1, 0).to(dev))
    assert torch.equal(dec_only.decode(z), img0)


def test_rejections(dev):
    from duodiff_b200._lib import DuoDiffError
    # in_channels > 7: conv_in's 9 * in_channels im2col columns do not fit one 64-wide K chunk
    wide = E.AEEncSpec(ch=64, ch_mult=[1, 2], num_res_blocks=1, resolution=32, in_channels=8)
    ae, _ = _make(wide, 0, 1)
    with pytest.raises(DuoDiffError, match="in_channels"):
        ae.encode_moments(torch.zeros(1, 8, 32, 32, device=dev))
    # the golden fixture's 32-channel toy geometry is below the kernel's 64-channel K chunk
    with pytest.raises(DuoDiffError, match="autoencoder:"):
        _make(E.AEEncSpec(ch=32, ch_mult=[1, 2, 2], num_res_blocks=1, resolution=32), 0, 1)
    # 2 * embed_dim moment planes must fit the 8-plane fp32 epilogue
    big_z = E.AEEncSpec(ch=64, ch_mult=[1, 2], num_res_blocks=1, resolution=32, z_channels=8, embed_dim=8)
    ae8, _ = _make(big_z, 0, 1)
    with pytest.raises(DuoDiffError, match="embed_dim"):
        ae8.encode_moments(torch.zeros(1, 3, 32, 32, device=dev))
    ae, _ = _make(SMALL, 0, 1)
    with pytest.raises(DuoDiffError, match="expects"):
        ae.encode_moments(torch.zeros(1, 3, 16, 16, device=dev))
    with pytest.raises(DuoDiffError, match="CUDA"):
        ae.encode_moments(torch.zeros(1, 3, 32, 32))
    with pytest.raises(DuoDiffError, match="CUDA"):
        ae.encode_moments(torch.zeros(1, 3, 32, 32, device=dev, dtype=torch.float16))
    with pytest.raises(DuoDiffError, match="expects"):
        ae.sample(torch.zeros(1, 4, 16, 16, device=dev))
