"""ctypes binding of include/duodiff_b200.h. No torch types cross this boundary: pointers, sizes, status codes."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

from ._build import LIB_PATH

_lib = None


class DuoDiffError(RuntimeError):
    pass


class UViTConfig(C.Structure):
    _fields_ = [
        ("img_size", C.c_int32), ("patch_size", C.c_int32), ("in_chans", C.c_int32), ("embed_dim", C.c_int32),
        ("depth", C.c_int32), ("num_heads", C.c_int32), ("mlp_hidden", C.c_int32), ("num_classes", C.c_int32),
        ("normalize_timesteps", C.c_int32), ("early_exit", C.c_int32), ("max_batch", C.c_int32),
        ("ln_eps", C.c_float),
    ]


class Tensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data_dev", C.c_void_p), ("numel", C.c_int64)]


class AEConfig(C.Structure):
    _fields_ = [
        ("ch", C.c_int32), ("out_ch", C.c_int32), ("num_res_blocks", C.c_int32), ("z_channels", C.c_int32),
        ("resolution", C.c_int32), ("embed_dim", C.c_int32), ("n_levels", C.c_int32), ("ch_mult", C.c_int32 * 8),
        ("max_batch", C.c_int32), ("scale_factor", C.c_float),
    ]


_P = C.c_void_p
_SIGS = {
    "ddb_version": (C.c_char_p, []),
    "ddb_last_error": (C.c_char_p, []),
    "ddb_launch_count": (C.c_int64, []),
    "ddb_model_create": (C.c_int, [C.POINTER(UViTConfig), C.POINTER(Tensor), C.c_int32, C.POINTER(_P)]),
    "ddb_model_destroy": (None, [_P]),
    "ddb_uvit_forward": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, _P]),
    "ddb_profile_forward": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, _P]),
    "ddb_ee_forward": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_float, C.c_int32, _P, _P, _P, _P, _P]),
    "ddb_ddpm_step": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, C.c_uint64, C.c_int64, _P]),
    "ddb_sampler_create": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, C.c_int32, C.c_float, C.c_int32,
                                     C.POINTER(_P)]),
    "ddb_sampler_destroy": (None, [_P]),
    "ddb_sampler_set_noise_offset": (C.c_int, [_P, C.c_uint64]),
    "ddb_sampler_set_guidance": (C.c_int, [_P, C.c_float, C.c_int64]),
    "ddb_sampler_profile_step": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "ddb_sampler_run": (C.c_int, [_P, _P, _P, _P, C.c_uint64, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_int32, _P]),
    "ddb_sampler_run_list": (C.c_int, [_P, _P, _P, _P, C.c_uint64, _P, _P, C.c_int32, _P, _P, C.c_int32, _P]),
    "ddb_sampler_run_list_logs": (C.c_int, [_P, _P, _P, _P, C.c_uint64, _P, _P, C.c_int32, _P, _P, _P, _P, C.c_int32,
                                            _P]),
    "ddb_finalize_nhwc": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "ddb_op_gemm": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, C.c_int32, C.c_int32,
                              C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "ddb_set_option": (C.c_int, [C.c_char_p, C.c_int32]),
    "ddb_debug_set_ptr": (C.c_int, [C.c_char_p, _P]),
    "ddb_op_attention": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "ddb_op_ln_stats": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P]),
    "ddb_ae_create": (C.c_int, [C.POINTER(AEConfig), C.POINTER(Tensor), C.c_int32, C.POINTER(_P)]),
    "ddb_ae_destroy": (None, [_P]),
    "ddb_ae_decode": (C.c_int, [_P, _P, C.c_int32, _P, _P]),
    "ddb_ae_profile_decode": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P]),
    "ddb_ae_num_ops": (C.c_int32, [_P]),
    "ddb_ae_op_info": (C.c_int, [_P, C.c_int32, C.c_char_p, C.c_int32, _P]),
    "ddb_ae_decode_debug": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int32, _P, _P]),
    "ddb_ae_create_encoder": (C.c_int, [_P, C.POINTER(Tensor), C.c_int32]),
    "ddb_ae_encode_moments": (C.c_int, [_P, _P, C.c_int32, _P, _P]),
    "ddb_ae_sample": (C.c_int, [_P, _P, _P, C.c_int32, _P, _P]),
    "ddb_ae_profile_encode": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P]),
    "ddb_ae_encoder_num_ops": (C.c_int32, [_P]),
    "ddb_ae_encoder_op_info": (C.c_int, [_P, C.c_int32, C.c_char_p, C.c_int32, _P]),
    "ddb_ae_encode_debug": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int32, _P, _P]),
    "ddb_op_pack_linear": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGS)


def load(path: Path | None = None):
    """Load libduodiff_b200.so. Fails loudly if it has not been built: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    p = Path(path or os.environ.get("DDB_LIB") or LIB_PATH)  # DDB_LIB: an A/B build (tools/, never the tests)
    if not p.exists():
        raise DuoDiffError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(duodiff_b200 has no CPU or PyTorch fallback)")
    lib = C.CDLL(str(p))
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        raise DuoDiffError(f"duodiff_b200 error {status}: {load().ddb_last_error().decode()}")


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def current_stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
