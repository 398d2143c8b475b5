"""ORACLE — test infrastructure only.  Never imported by the product path (duodiff_b200/).

Functional fp32 restatement of the encode side of ``FrozenAutoencoderKL`` (``encode_moments`` = ``quant_conv`` after
``Encoder.forward``, the DiagonalGaussian ``sample``, ``encode`` = ``sample(encode_moments(x))``), operating directly on
a reference ``state_dict``.  ``encode_moments`` can return the named intermediate tensors the CUDA path exposes through
``ddb_ae_encode_debug`` (the encoder's op names) so that a parity failure can be localised to one layer.

The blocks it shares with the decoder (``resnet_block``, ``attn_block``, ``_gn`` of ``oracle/ae_oracle.py``) are pinned
to the reference by ``tests/golden/ae_decode_tiny.npz``.  The encoder's own wiring -- the level loop with
``num_res_blocks`` blocks per level, the asymmetrically padded stride-2 Downsample, conv_out with ``double_z``,
quant_conv and the sample formula -- is restated from the reference's module and is NOT pinned by a fixture made from
the reference itself.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from oracle.ae_oracle import AESpec, _conv, _gn, _swish, attn_block, resnet_block


@dataclass
class AEEncSpec(AESpec):
    """ddconfig of get_autoencoder plus what only the encoder reads (Encoder.__init__: in_channels)."""
    in_channels: int = 3


def encode_moments(sd: Dict[str, torch.Tensor], spec: AEEncSpec, x: torch.Tensor,
                   tap: Optional[dict] = None) -> torch.Tensor:
    """FrozenAutoencoderKL.encode_moments = quant_conv(Encoder.forward(x)): x [B, in_channels, res, res] ->
    moments [B, 2*embed_dim, z_res, z_res].  ``tap`` receives the NCHW intermediates under the encoder op names."""
    sd = {k: v.float() for k, v in sd.items()}
    h = _conv(sd, "encoder.conv_in", x.float(), 1)
    if tap is not None:
        tap["conv_in"] = h
    n_levels = len(spec.ch_mult)
    for lvl in range(n_levels):
        for j in range(spec.num_res_blocks):  # num_res_blocks per level (the decoder has one more)
            h = resnet_block(sd, f"encoder.down.{lvl}.block.{j}", h, tap, f"down.{lvl}.block.{j}")
        if lvl != n_levels - 1:  # Downsample(with_conv=True): pad right / bottom by one, 3x3 conv, stride 2
            h = F.conv2d(F.pad(h, (0, 1, 0, 1), mode="constant", value=0),
                         sd[f"encoder.down.{lvl}.downsample.conv.weight"],
                         sd[f"encoder.down.{lvl}.downsample.conv.bias"], stride=2, padding=0)
            if tap is not None:
                tap[f"down.{lvl}.downsample"] = h
    h = resnet_block(sd, "encoder.mid.block_1", h, tap, "mid.block_1")
    h = attn_block(sd, "encoder.mid.attn_1", h, tap, "mid.attn_1")
    h = resnet_block(sd, "encoder.mid.block_2", h, tap, "mid.block_2")
    h = _swish(_gn(sd, "encoder.norm_out", h))
    if tap is not None:
        tap["norm_out"] = h
    h = _conv(sd, "encoder.conv_out", h, 1)  # -> 2 * z_channels (double_z)
    moments = _conv(sd, "quant_conv", h, 0)
    if tap is not None:
        tap["moments"] = moments
    return moments


def sample(moments: torch.Tensor, noise: torch.Tensor, scale: float) -> torch.Tensor:
    """FrozenAutoencoderKL.sample: z = scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise)."""
    mean, logvar = torch.chunk(moments, 2, dim=1)
    logvar = torch.clamp(logvar, -30.0, 20.0)
    std = torch.exp(0.5 * logvar)
    return scale * (mean + std * noise)


def random_encoder_state_dict(spec: AEEncSpec, seed: int, hot: bool = True) -> Dict[str, torch.Tensor]:
    """Encoder-side state_dict (``encoder.*``, ``quant_conv.*``) with the reference's key names and shapes
    (Encoder.__init__, quant_conv of FrozenAutoencoderKL.__init__); same initialisation as ``random_state_dict``."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}

    def conv(key, cout, cin, k, gain=1.0):
        fan = cin * k * k
        sd[key + ".weight"] = torch.randn(cout, cin, k, k, generator=g) * (gain / fan ** 0.5)
        sd[key + ".bias"] = torch.randn(cout, generator=g) * (0.1 if hot else 0.0)

    def norm(key, c):
        sd[key + ".weight"] = 1.0 + (torch.randn(c, generator=g) * 0.2 if hot else torch.zeros(c))
        sd[key + ".bias"] = torch.randn(c, generator=g) * 0.2 if hot else torch.zeros(c)

    def res(key, cin, cout):
        norm(key + ".norm1", cin)
        conv(key + ".conv1", cout, cin, 3, 1.4)
        norm(key + ".norm2", cout)
        conv(key + ".conv2", cout, cout, 3, 0.7)
        if cin != cout:
            conv(key + ".nin_shortcut", cout, cin, 1)

    n = len(spec.ch_mult)
    conv("encoder.conv_in", spec.ch, spec.in_channels, 3)
    c = spec.ch
    for lvl in range(n):
        co = spec.ch * spec.ch_mult[lvl]
        for j in range(spec.num_res_blocks):
            res(f"encoder.down.{lvl}.block.{j}", c, co)
            c = co
        if lvl != n - 1:
            conv(f"encoder.down.{lvl}.downsample.conv", c, c, 3)
    res("encoder.mid.block_1", c, c)
    norm("encoder.mid.attn_1.norm", c)
    for s in ("q", "k", "v", "proj_out"):
        conv(f"encoder.mid.attn_1.{s}", c, c, 1, 1.5 if s in ("q", "k") else 1.0)
    res("encoder.mid.block_2", c, c)
    norm("encoder.norm_out", c)
    conv("encoder.conv_out", 2 * spec.z_channels, c, 3)
    conv("quant_conv", 2 * spec.embed_dim, 2 * spec.z_channels, 1)
    return sd
