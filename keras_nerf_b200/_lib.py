"""ctypes binding of libknerf.so (C ABI declared in include/knerf.h).

This is the only place Python touches native code.  There is NO CPU fallback: if the shared library
is missing or a tensor is not on a CUDA device the call fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# KNERF_LIB_PATH: diagnostics only (e.g. a -DKNERF_TC_TIMING build kept next to the release library)
LIB_PATH = os.environ.get("KNERF_LIB_PATH") or os.path.join(_HERE, "lib", "libknerf.so")

OOB_ZERO, OOB_CLAMP, OOB_COUNT = 0, 1, 2
SCAN_SEQUENTIAL = 0x10   # OR-ed into oob_mode: pdf/cdf summed left to right (TF-CPU / NumPy order)
FP32, BF16, FP32_TC = 0, 1, 2
# per-call option bits OR-ed into `precision` (include/knerf.h)
PRECISION_MASK, TC_ORDERED, BWD_DGRAD_ONLY, BWD_WGRAD_ONLY, REC_FP8 = 0xFF, 0x100, 0x200, 0x400, 0x800
COMM_ID_BYTES = 128
PRECISIONS = {"fp32": FP32, "float32": FP32, "bf16": BF16, "bfloat16": BF16, "fp32_tc": FP32_TC, "fp32tc": FP32_TC}
OOB_MODES = {"zero": OOB_ZERO, "clamp": OOB_CLAMP, "raise": OOB_COUNT}


class KnerfError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_coarse", "n_fine", "pos_emb_xyz", "pos_emb_dir", "n_layers",
                                         "dense_units", "skip_layer", "dx", "dd")]


_P, _I, _L, _F, _U64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64
_CFG = C.POINTER(Config)

# name -> (restype, argtypes); must list every symbol include/knerf.h and include/knerf_debug.h declare (tests check
# this)
SIGNATURES = {
    "knerf_abi_version": (_I, []),
    "knerf_last_error": (C.c_char_p, []),
    "knerf_launch_count": (_U64, []),
    "knerf_device_supports_bf16": (_I, []),
    "knerf_generate_rays": (_I, [_P, _I, _I, _F, _F, _F, _I, _P, _U64, _P, _P, _P, _P]),
    "knerf_generate_ray_batch": (_I, [_P, _I, _I, _I, _I, _P, _F, _F, _F, _I, _U64, _U64, _L, _L, _P, _U64,
                                      _P, _P, _P, _P, _P, _P]),
    "knerf_uniform": (_I, [_P, _L, _U64, _U64, _P]),
    "knerf_positional_encoding": (_I, [_P, _L, _I, _I, _P, _I, _P]),
    "knerf_encode_position_and_directions": (_I, [_P, _P, _P, _L, _I, _I, _I, _P, _I, _P, _I, _P]),
    "knerf_composite_forward": (_I, [_P, _P, _P, _P, _L, _I, _I, _I, _F, _P, _P, _P, _P, _P]),
    "knerf_composite_backward": (_I, [_P, _P, _L, _I, _I, _I, _F, _P, _P, _F, _I, _P, _P, _P]),
    "knerf_sample_fine": (_I, [_P, _P, _P, _P, _U64, _P, _L, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
    "knerf_param_count": (_L, [_CFG]),
    "knerf_layer_table": (_I, [_CFG, _I, _P, _P, _P, _P]),
    "knerf_workspace_bytes": (_L, [_CFG, _L, _I, _I]),
    "knerf_mlp_forward_encoded": (_I, [_CFG, _P, _P, _I, _P, _I, _L, _P, _P, _P, _L, _P]),
    "knerf_packed_weight_bytes": (_L, [_CFG]),
    "knerf_pack_weights": (_I, [_CFG, _P, _P, _P]),
    "knerf_mlp_forward": (_I, [_CFG, _P, _P, _P, _P, _P, _L, _I, _I, _I, _P, _P, _L, _P]),
    "knerf_mlp_backward": (_I, [_CFG, _P, _P, _P, _L, _I, _I, _P, _P, _L, _P]),
    "knerf_render_chunk": (_I, [_CFG, _P, _P, _P, _P, _P, _P, _P, _L, _P, _U64, _I, _I, _I,
                                _P, _P, _P, _P, _P, _P, _P, _P, _L, _P]),
    "knerf_train_chunk": (_I, [_CFG, _P, _P, _P, _P, _P, _P, _P, _P, _L, _P, _U64, _I, _I, _I, _F,
                               _P, _P, _P, _P, _P, _P, _L, _P]),
    "knerf_adam_step": (_I, [_P, _P, _P, _P, _L, _F, _F, _F, _F, _L, _I, _P]),
    "knerf_mse": (_I, [_P, _P, _L, _P, _P]),
    "knerf_image_prepare": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "knerf_image_metrics_workspace_floats": (_L, [_I, _I, _I, _I]),
    "knerf_image_metrics": (_I, [_P, _P, _I, _I, _I, _I, _F, _P, _P, _P, _L, _P]),
    "knerf_comm_unique_id": (_I, [_P]),
    "knerf_comm_create": (_I, [_P, _I, _I, C.POINTER(_P)]),
    "knerf_comm_adopt": (_I, [_P, _I, _I, C.POINTER(_P)]),
    "knerf_comm_destroy": (_I, [_P]),
    "knerf_comm_rank": (_I, [_P, C.POINTER(_I), C.POINTER(_I)]),
    "knerf_allreduce_grads": (_I, [_P, _P, _L, _P]),
    "knerf_train_chunk_dp": (_I, [_CFG, _P, _P, _P, _P, _P, _P, _P, _P, _L, _P, _U64, _I, _I, _I, _F,
                                  _P, _P, _P, _P, _P, _P, _L, _P, _P, _P, _I]),
    "knerf_isosurface_workspace_bytes": (_L, [_I, _I, _I]),
    "knerf_isosurface_count": (_I, [_P, _I, _I, _I, _F, _P, _P, _L, _P]),
    "knerf_isosurface_emit": (_I, [_P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _L, _L, _P, _L, _P]),
    "knerf_debug_tc_timing": (_I, [_P, _I]),
    "knerf_debug_wgrad_timing": (_I, [_P, _I]),
    "knerf_debug_dgrad_timing": (_I, [_P, _I]),
    "knerf_selftest_umma": (_I, [_I, _P, _P, _I, _I, _P, _P]),
    "knerf_selftest_umma2": (_I, [_P, _P, _I, _I, _P, _P]),
}

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(keras_nerf_b200 has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.knerf_abi_version() != 2:
            raise ImportError("libknerf.so ABI version mismatch")
        _lib = lib
    return _lib


def check(status: int) -> None:
    if status != 0:
        raise KnerfError(f"libknerf error {status}: {load().knerf_last_error().decode()}")


def call(name: str, *args):
    """Invoke an int-status entry point and raise on error."""
    check(getattr(load(), name)(*args))


def ptr(t: Optional[torch.Tensor], dtype=torch.float32) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise KnerfError("libknerf needs CUDA tensors (no CPU fallback)")
    if t.dtype != dtype or not t.is_contiguous():
        raise KnerfError(f"expected contiguous {dtype} tensor, got {t.dtype} contiguous={t.is_contiguous()}")
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def dev(x, device, dtype=torch.float32) -> torch.Tensor:
    """numpy / torch / any DLPack producer (tf.Tensor via tf.experimental.dlpack, cupy, jax ...; any device) ->
    contiguous tensor on `device`.  A DLPack producer that already lives on `device` is consumed zero-copy: this is
    the shim a TensorFlow caller goes through (INTEGRATION.md)."""
    if not torch.is_tensor(x) and hasattr(x, "__dlpack__") and not hasattr(x, "__array_interface__"):
        x = torch.from_dlpack(x)
    return torch.as_tensor(x, dtype=dtype, device=device).contiguous()


def seed_stream(tag: int, advance: int = 0):
    """Philox seed stream of this process for draws the caller did not pin (`seed=None`): an `itertools.count` keyed
    by `tag` (which generator), the torch seed (torch.manual_seed; the scripts' tf.random.set_seed) and the RANK, so
    the replicas of a data-parallel run draw independent samples (every replica of a MirroredStrategy has its own
    tf.random stream too); `advance` skips ahead (a resumed run must not replay epoch 0's draws)."""
    import itertools
    rank = int(os.environ.get("RANK", "0"))
    base = (tag + (torch.initial_seed() & 0xFFFFFFFF) * 0x9E3779B1 + rank * 0x9E3779B97F4A7C15
            + advance * 0x632BE59BD9B4E019)
    return itertools.count(base & 0x3FFFFFFFFFFFFFFF)


def default_device() -> torch.device:
    if not torch.cuda.is_available():
        raise KnerfError("keras_nerf_b200 needs a CUDA device (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())
