"""Drop-in for the reference's ``models/utils/autoencoder.py`` (``FrozenAutoencoderKL`` :452-500, ``get_autoencoder``
:503-516): the latent -> image decoder that ``sampler.get_samples`` / ``eesampler.get_samples`` call after the last
denoising step of a latent model (sampler.py:141-143, eesampler.py:84-85), and the image -> latent encoder
(``encode_moments`` / ``sample`` / ``encode``) used to prepare latents and to check reconstructions.

All arithmetic runs inside libduodiff_b200.so (implicit-GEMM tcgen05 convolutions, csrc/conv_gemm.cuh); PyTorch only
owns the device memory (and draws the sampling noise).  The encoder is built on the first encode call, so callers that
only decode pay nothing for it.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import torch

from . import _lib

# ddconfig of get_autoencoder (models/utils/autoencoder.py:504-515)
DEFAULT_DDCONFIG = dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128,
                        ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0)


class FrozenAutoencoderKL:
    """``FrozenAutoencoderKL(ddconfig, embed_dim, pretrained_path, scale_factor)`` (autoencoder.py:452-466).

    ``pretrained_path`` is a ``torch.save``d state_dict with the reference's keys; ``state_dict=`` hands the tensors
    over directly (tests, random-init throughput runs).  ``max_batch`` is the number of latents decoded per pass
    (larger batches are processed in chunks)."""

    PROF_CATEGORIES = ("conv3x3", "conv_upsample", "conv1x1", "attn_matmul", "groupnorm", "other")

    def __init__(self, ddconfig: dict, embed_dim: int, pretrained_path: Optional[str] = None,
                 scale_factor: float = 0.18215, *, state_dict: Optional[Dict[str, torch.Tensor]] = None,
                 max_batch: int = 16):
        if ddconfig.get("attn_resolutions"):
            raise NotImplementedError("attn_resolutions != [] (the reference's get_autoencoder uses [])")
        if ddconfig.get("use_linear_attn") or ddconfig.get("attn_type", "vanilla") != "vanilla":
            raise NotImplementedError("only attn_type='vanilla' (the reference default) is supported")
        if ddconfig.get("tanh_out") or ddconfig.get("give_pre_end"):
            raise NotImplementedError("tanh_out / give_pre_end are not used by the reference's sampler")
        assert ddconfig.get("double_z", True)  # autoencoder.py:458
        if state_dict is None:
            if pretrained_path is None:
                raise ValueError("either pretrained_path or state_dict is required")
            state_dict = torch.load(pretrained_path, map_location="cpu")
        if not torch.cuda.is_available():
            raise _lib.DuoDiffError("duodiff_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        print(f"Create autoencoder with scale_factor={scale_factor}")
        self.lib = _lib.load()
        self.ddconfig = dict(ddconfig)
        self.embed_dim = embed_dim
        self.scale_factor = scale_factor
        self.z_channels = int(ddconfig["z_channels"])
        self.out_ch = int(ddconfig["out_ch"])
        self.resolution = int(ddconfig["resolution"])
        mult: Sequence[int] = ddconfig["ch_mult"]
        self.z_res = self.resolution // 2 ** (len(mult) - 1)
        self.in_channels = int(ddconfig.get("in_channels", 3))
        self.cfg = _lib.AEConfig(int(ddconfig["ch"]), self.out_ch, int(ddconfig["num_res_blocks"]), self.z_channels,
                                 self.resolution, int(embed_dim), len(mult),
                                 (C.c_int32 * 8)(*[int(m) for m in mult]), int(max_batch), float(scale_factor))
        dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        used = {k: v for k, v in state_dict.items() if k.startswith("decoder.") or k.startswith("post_quant_conv.")}
        with torch.cuda.device(dev):
            keep, arr = [], (_lib.Tensor * len(used))()
            for i, (name, t) in enumerate(used.items()):
                t = t.detach().to(device=dev, dtype=torch.float32).contiguous()
                keep.append(t)
                arr[i] = _lib.Tensor(name.encode(), t.data_ptr(), t.numel())
            torch.cuda.synchronize(dev)
            handle = C.c_void_p()
            _lib.check(self.lib.ddb_ae_create(C.byref(self.cfg), arr, len(used), C.byref(handle)))
            self.handle = handle
            del keep
        # encoder weights stay on the host until the first encode call (see _encoder)
        self._enc_sd = {k: v for k, v in state_dict.items()
                        if k.startswith("encoder.") or k.startswith("quant_conv.")}
        self._enc_built = False

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            try:
                with torch.cuda.device(self.device):
                    self.lib.ddb_ae_destroy(h)
            except (AttributeError, TypeError):  # interpreter shutdown: torch is already torn down
                pass
            self.handle = None

    # nn.Module surface the reference's callers touch
    def eval(self):
        return self

    def to(self, *_a, **_k):
        return self

    def requires_grad_(self, *_a, **_k):
        return self

    def _check_cuda(self, t, what, shape):
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.dim() == 4):
            raise _lib.DuoDiffError(f"{what} must be a CUDA float32 tensor [B, {shape[0]}, {shape[1]}, {shape[2]}]")
        if t.device != self.device:
            raise _lib.DuoDiffError(f"{what} is on {t.device} but the autoencoder lives on {self.device}")
        if tuple(t.shape[1:]) != tuple(shape):
            raise _lib.DuoDiffError(f"{what} has shape {tuple(t.shape)}, autoencoder expects "
                                    f"[B,{shape[0]},{shape[1]},{shape[2]}]")
        return t.contiguous()

    def _check(self, z):
        return self._check_cuda(z, "z", (self.z_channels, self.z_res, self.z_res))

    def decode(self, z: torch.Tensor) -> torch.Tensor:
        """autoencoder.py:486-490: ``decoder(post_quant_conv(z / scale_factor))`` -> [B, out_ch, res, res] fp32."""
        z = self._check(z)
        out = torch.empty(z.shape[0], self.out_ch, self.resolution, self.resolution, device=z.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_ae_decode(self.handle, z.data_ptr(), z.shape[0], out.data_ptr(),
                                              _lib.current_stream_ptr()))
        return out

    def forward(self, inputs, fn):  # autoencoder.py:492-500
        if fn == "encode_moments":
            return self.encode_moments(inputs)
        elif fn == "encode":
            return self.encode(inputs)
        elif fn == "decode":
            return self.decode(inputs)
        raise NotImplementedError

    __call__ = forward

    # ------------------------------------------------------------------ encode side
    def _encoder(self):
        """Build the encoder plan on the first encode call from the ``encoder.*`` / ``quant_conv.*`` tensors kept at
        construction (a missing key raises DuoDiffError naming it)."""
        if self._enc_built:
            return
        w = self._enc_sd.get("encoder.conv_in.weight")
        if w is not None and w.dim() == 4 and int(w.shape[1]) != self.in_channels:
            raise _lib.DuoDiffError(f"encoder.conv_in.weight has {int(w.shape[1])} input channels, ddconfig "
                                    f"in_channels is {self.in_channels}")
        with torch.cuda.device(self.device):
            keep, arr = [], (_lib.Tensor * max(len(self._enc_sd), 1))()
            for i, (name, t) in enumerate(self._enc_sd.items()):
                t = t.detach().to(device=self.device, dtype=torch.float32).contiguous()
                keep.append(t)
                arr[i] = _lib.Tensor(name.encode(), t.data_ptr(), t.numel())
            torch.cuda.synchronize(self.device)
            _lib.check(self.lib.ddb_ae_create_encoder(self.handle, arr, len(self._enc_sd)))
            del keep
        self._enc_built = True
        self._enc_sd = {}  # packed on the device now

    def _check_image(self, x):
        return self._check_cuda(x, "x", (self.in_channels, self.resolution, self.resolution))

    def _moments_out(self, x):
        return torch.empty(x.shape[0], 2 * self.embed_dim, self.z_res, self.z_res, device=x.device)

    def encode_moments(self, x: torch.Tensor) -> torch.Tensor:
        """``quant_conv(encoder(x))``: x [B, in_channels, res, res] fp32 -> moments [B, 2*embed_dim, r, r] fp32."""
        x = self._check_image(x)
        self._encoder()
        out = self._moments_out(x)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_ae_encode_moments(self.handle, x.data_ptr(), x.shape[0], out.data_ptr(),
                                                      _lib.current_stream_ptr()))
        return out

    def sample(self, moments: torch.Tensor, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``scale_factor * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise)`` with ``mean, logvar =
        chunk(moments, 2, dim=1)``; ``noise=None`` draws ``torch.randn_like(mean)`` as the reference does."""
        moments = self._check_cuda(moments, "moments", (2 * self.embed_dim, self.z_res, self.z_res))
        if noise is None:
            mean, _logvar = torch.chunk(moments, 2, dim=1)
            noise = torch.randn_like(mean)
        noise = self._check_cuda(noise, "noise", (self.embed_dim, self.z_res, self.z_res))
        if noise.shape[0] != moments.shape[0]:
            raise _lib.DuoDiffError(f"noise has batch {noise.shape[0]}, moments {moments.shape[0]}")
        z = torch.empty(moments.shape[0], self.embed_dim, self.z_res, self.z_res, device=moments.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_ae_sample(self.handle, moments.data_ptr(), noise.data_ptr(), moments.shape[0],
                                              z.data_ptr(), _lib.current_stream_ptr()))
        return z

    def encode(self, x: torch.Tensor, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``sample(encode_moments(x))``: x [B, in_channels, res, res] -> z [B, embed_dim, r, r] (scaled latents)."""
        return self.sample(self.encode_moments(x), noise)

    # ------------------------------------------------------------------ measurement / parity hooks
    def profile_decode(self, z: torch.Tensor) -> dict:
        z = self._check(z)
        out = torch.empty(z.shape[0], self.out_ch, self.resolution, self.resolution, device=z.device)
        n = len(self.PROF_CATEGORIES)
        ms, fl = (C.c_float * n)(), (C.c_double * n)()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_ae_profile_decode(self.handle, z.data_ptr(), z.shape[0], out.data_ptr(), ms, fl,
                                                      _lib.current_stream_ptr()))
        return {k: dict(ms=float(ms[i]), flops=float(fl[i])) for i, k in enumerate(self.PROF_CATEGORIES)}

    def _op_list(self, num_ops, op_info):
        res = []
        for i in range(num_ops(self.handle)):
            name, info = C.create_string_buffer(96), (C.c_int32 * 4)()
            _lib.check(op_info(self.handle, i, name, 96, info))
            res.append((name.value.decode(), *[int(v) for v in info]))
        return res

    def ops(self):
        """[(name, C, H, W, is_f32)] of the launch list (C == 0: the op leaves nothing to dump)."""
        return self._op_list(self.lib.ddb_ae_num_ops, self.lib.ddb_ae_op_info)

    def decode_debug(self, z: torch.Tensor, op_index: int):
        """(image, NCHW fp32 copy of op `op_index`'s output) for z with B <= max_batch."""
        z = self._check(z)
        name, c, h, w, f32 = self.ops()[op_index]
        out = torch.empty(z.shape[0], self.out_ch, self.resolution, self.resolution, device=z.device)
        dump = torch.empty(z.shape[0], h, w, c, device=z.device, dtype=torch.float32 if f32 else torch.bfloat16)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_ae_decode_debug(self.handle, z.data_ptr(), z.shape[0], out.data_ptr(), op_index,
                                                    dump.data_ptr(), _lib.current_stream_ptr()))
        return out, dump.float().permute(0, 3, 1, 2).contiguous()


    def profile_encode(self, x: torch.Tensor) -> dict:
        x = self._check_image(x)
        self._encoder()
        out = self._moments_out(x)
        n = len(self.PROF_CATEGORIES)
        ms, fl = (C.c_float * n)(), (C.c_double * n)()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_ae_profile_encode(self.handle, x.data_ptr(), x.shape[0], out.data_ptr(), ms, fl,
                                                      _lib.current_stream_ptr()))
        return {k: dict(ms=float(ms[i]), flops=float(fl[i])) for i, k in enumerate(self.PROF_CATEGORIES)}

    def encoder_ops(self):
        """[(name, C, H, W, is_f32)] of the encoder's launch list (builds the encoder)."""
        self._encoder()
        return self._op_list(self.lib.ddb_ae_encoder_num_ops, self.lib.ddb_ae_encoder_op_info)

    def encode_debug(self, x: torch.Tensor, op_index: int):
        """(moments, NCHW fp32 copy of encoder op `op_index`'s output) for x with B <= max_batch."""
        x = self._check_image(x)
        name, c, h, w, f32 = self.encoder_ops()[op_index]
        out = self._moments_out(x)
        dump = torch.empty(x.shape[0], h, w, c, device=x.device, dtype=torch.float32 if f32 else torch.bfloat16)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ddb_ae_encode_debug(self.handle, x.data_ptr(), x.shape[0], out.data_ptr(), op_index,
                                                    dump.data_ptr(), _lib.current_stream_ptr()))
        return out, dump.float().permute(0, 3, 1, 2).contiguous()

def random_init_state_dict(ddconfig: dict = DEFAULT_DDCONFIG, embed_dim: int = 4, seed: int = 0, encoder: bool = False):
    """Decoder-side state_dict with the reference's keys and shapes (Decoder.__init__, autoencoder.py:320-412) and
    PyTorch's default Conv2d / GroupNorm initialisation -- for throughput runs, since no autoencoder checkpoint ships
    with the reference (SURVEY.md §8d: random-init weights of the configured architecture).  ``encoder=True`` adds the
    ``encoder.*`` / ``quant_conv.*`` keys (drawn after the decoder's, which stay the same)."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}

    def conv(key, cout, cin, k):
        bound = 1.0 / (cin * k * k) ** 0.5  # kaiming_uniform(a=sqrt(5)) and the bias bound coincide
        sd[key + ".weight"] = (torch.rand(cout, cin, k, k, generator=g) * 2 - 1) * bound
        sd[key + ".bias"] = (torch.rand(cout, generator=g) * 2 - 1) * bound

    def norm(key, c):
        sd[key + ".weight"], sd[key + ".bias"] = torch.ones(c), torch.zeros(c)

    def res(key, cin, cout):
        norm(key + ".norm1", cin)
        conv(key + ".conv1", cout, cin, 3)
        norm(key + ".norm2", cout)
        conv(key + ".conv2", cout, cout, 3)
        if cin != cout:
            conv(key + ".nin_shortcut", cout, cin, 1)

    mult, ch, zc = ddconfig["ch_mult"], ddconfig["ch"], ddconfig["z_channels"]
    conv("post_quant_conv", zc, embed_dim, 1)
    c = ch * mult[-1]
    conv("decoder.conv_in", c, zc, 3)
    res("decoder.mid.block_1", c, c)
    norm("decoder.mid.attn_1.norm", c)
    for name in ("q", "k", "v", "proj_out"):
        conv(f"decoder.mid.attn_1.{name}", c, c, 1)
    res("decoder.mid.block_2", c, c)
    for lvl in reversed(range(len(mult))):
        co = ch * mult[lvl]
        for j in range(ddconfig["num_res_blocks"] + 1):
            res(f"decoder.up.{lvl}.block.{j}", c, co)
            c = co
        if lvl != 0:
            conv(f"decoder.up.{lvl}.upsample.conv", c, c, 3)
    norm("decoder.norm_out", c)
    conv("decoder.conv_out", ddconfig["out_ch"], c, 3)
    if not encoder:
        return sd
    c = ch
    conv("encoder.conv_in", c, ddconfig.get("in_channels", 3), 3)
    for lvl in range(len(mult)):
        co = ch * mult[lvl]
        for j in range(ddconfig["num_res_blocks"]):
            res(f"encoder.down.{lvl}.block.{j}", c, co)
            c = co
        if lvl != len(mult) - 1:
            conv(f"encoder.down.{lvl}.downsample.conv", c, c, 3)
    res("encoder.mid.block_1", c, c)
    norm("encoder.mid.attn_1.norm", c)
    for name in ("q", "k", "v", "proj_out"):
        conv(f"encoder.mid.attn_1.{name}", c, c, 1)
    res("encoder.mid.block_2", c, c)
    norm("encoder.norm_out", c)
    conv("encoder.conv_out", 2 * zc, c, 3)
    conv("quant_conv", 2 * embed_dim, 2 * zc, 1)
    return sd


def get_autoencoder(pretrained_path, scale_factor=0.18215, *, max_batch: int = 16):
    """models/utils/autoencoder.py:503-516."""
    return FrozenAutoencoderKL(DEFAULT_DDCONFIG, 4, pretrained_path, scale_factor, max_batch=max_batch)
