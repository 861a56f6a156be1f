"""ctypes binding of libaa_b200.so (include/aa_b200.h).  No torch types cross this boundary:
only raw device pointers, sizes, strides, scalars and the stream handle.

There is NO CPU fallback: if the library cannot be loaded (or built with nvcc when absent),
importing the compute path raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_uint32, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('AA_B200_LIB') or os.path.join(_HERE, 'csrc', 'libaa_b200.so')

AA_BF16, AA_F16, AA_F32 = 0, 1, 2
MODE_FAITHFUL, MODE_F32, MODE_CE = 0, 1, 2  # MODE_CE: K6 / K6b only (include/aa_b200.h)
MASK_U8, MASK_I64 = 0, 1
STATUS_LABEL_OOB, STATUS_SHORT_SEQUENCE, STATUS_EMPTY_MASK, STATUS_DIVERGE_RANGE = 1, 2, 4, 8

_DTYPE_CODE = {torch.bfloat16: AA_BF16, torch.float16: AA_F16, torch.float32: AA_F32}
_CODE_DTYPE = {v: k for k, v in _DTYPE_CODE.items()}

_lib = None


class AaColl(Structure):
    """include/aa_b200.h `aa_coll`: descriptor of the one-shot NVLink all-reduce."""

    _fields_ = [('peer_bufs', c_void_p), ('rank', c_int32), ('world', c_int32), ('epoch', c_uint32),
                ('max_lanes', c_uint32)]


_P = c_void_p
_SIGS = {
    'aa_abi_version': (c_int, []),
    'aa_last_error': (c_char_p, []),
    'aa_device_info': (c_int, [POINTER(c_int), POINTER(c_int)]),
    'aa_logprob_set_tuning': (c_int, [c_int, c_int]),
    'aa_logprob_set_tuning_bwd': (c_int, [c_int, c_int]),
    'aa_logprob_fwd': (c_int, [_P, c_int, c_int64, c_int32, _P, c_int64, c_int32, c_int32, c_int64, _P, _P, _P, _P,
                               _P, c_int, _P, _P, _P, _P]),
    'aa_logprob_bwd': (c_int, [_P, c_int, c_int64, c_int32, _P, c_int64, c_int32, c_int32, c_int64, _P, _P, _P, _P,
                               _P, _P, _P, _P, c_int, _P, _P, c_int, _P, c_int64, c_int64, _P, c_int64, _P, c_int, _P]),
    'aa_zero_rows': (c_int, [_P, c_int, c_int64, c_int32, c_int64, _P, c_int32, _P]),
    'aa_linear_dlogits': (c_int, [_P, c_int64, c_int32, c_int64, _P, c_int32, c_int64, _P, _P, _P, _P, c_int, _P, c_int64, c_int, _P]),
    'aa_linear_dhidden': (c_int, [_P, c_int64, c_int64, _P, c_int32, c_int32, c_int64, _P, c_int64, _P]),
    'aa_linear_dweight': (c_int, [_P, c_int64, c_int64, _P, c_int32, c_int64, c_int32, _P, c_int64, c_int32, _P, c_int64, _P]),
    'aa_linear_logprob_fwd': (c_int, [_P, c_int64, c_int32, c_int64, _P, c_int32, c_int64, _P, _P, c_int, _P, _P, _P, c_int64,
                                      c_int, _P, _P]),
    'aa_strip_pad_tail': (c_int, [_P, c_int32, c_int32, c_int64, c_int64, c_int, _P, _P, c_int64, _P, _P]),
    'aa_dpo_loss': (c_int, [_P, _P, c_int, c_int32, c_int32, c_int64, c_float, c_int, _P, c_int32, c_int64,
                            _P, _P, _P, _P, POINTER(AaColl), _P, _P, _P]),
    'aa_pair_slices': (c_int, [_P, c_int64, _P, c_int, c_int64, c_int32, c_int32, _P, _P, _P]),
    'aa_slice_sums': (c_int, [_P, c_int, c_int64, c_int32, c_int32, _P, c_int, _P, _P]),
    'aa_rm_pair_loss': (c_int, [_P, c_int32, c_float, _P, _P, _P]),
    'aa_score_head_fwd': (c_int, [_P, c_int, c_int64, c_int32, c_int64, _P, _P, c_int, c_int, _P]),
    'aa_score_end': (c_int, [_P, c_int, c_int64, _P, c_int, c_int64, c_int32, c_int32, _P, _P, _P, c_int,
                             c_int64, c_int64, c_int32, _P, _P, _P]),
    'aa_score_head_bwd': (c_int, [_P, c_int, c_int64, c_int32, c_int64, _P, _P, c_int, _P, c_int64, _P, _P,
                                  POINTER(c_int32), c_int, _P]),
    'aa_ppo_prep': (c_int, [_P, _P, c_int, c_int64, _P, _P, c_int, c_int64, _P, c_int64, c_int32, c_int32,
                            c_int32, c_float, c_float, c_float, c_float, c_int, _P, c_int, _P, _P, c_int, _P,
                            _P, _P]),
    'aa_ppo_actor_loss': (c_int, [_P, c_int64, _P, c_int64, c_int, _P, c_int64, c_int, _P, c_int64, c_int32,
                                  c_int32, c_float, c_int, _P, _P, c_int64, _P, _P, _P]),
    'aa_ppo_critic_loss': (c_int, [_P, c_int64, _P, c_int64, c_int, _P, c_int64, c_int, _P, c_int64, c_int32,
                                   c_int32, c_float, c_int, _P, _P, c_int64, _P, _P, _P, _P, c_int32, _P]),
    'aa_logprob_actor_fused': (c_int, [_P, c_int, c_int64, c_int32, _P, c_int32, _P, _P, _P, _P, _P, c_int64, _P, c_int, _P, _P,
                                       _P, c_int64, _P, c_int64, c_int, _P, c_int64, c_int32, c_float, c_int, _P, c_int64, _P,
                                       _P, _P]),
    'aa_logprob_ce_fused': (c_int, [_P, c_int, c_int64, c_int32, _P, c_int64, c_int64, c_int32, _P, _P, _P, _P, _P, c_int64, _P,
                                    c_float, _P, c_int64, _P, _P, _P, _P]),
    'aa_logprob_grpo_fused': (c_int, [_P, c_int, c_int64, c_int32, _P, c_int32, _P, _P, _P, _P, _P, c_int64, _P, c_int, _P, c_int64,
                                      _P, _P, c_int64, c_int64, c_int32, c_float, c_int, _P, c_int64, _P, _P, _P, _P, _P, _P]),
    'aa_scale_tile': (c_int, [_P, c_int, c_int64, _P, c_int, _P]),
    'aa_tail_scatter_scaled': (c_int, [_P, c_int, c_int64, _P, c_int32, c_int32, c_int32, _P, c_int, _P, c_int64, c_int32, _P]),
    'aa_group_advantages': (c_int, [_P, c_int32, c_int32, _P, _P]),
    'aa_grpo_loss': (c_int, [_P, c_int64, _P, c_int64, c_int, _P, _P, c_int64, c_int64, c_int32, c_int32, c_float, c_int,
                             _P, _P, c_int64, _P, _P, _P, _P]),
    'aa_nll_mean': (c_int, [_P, c_int, _P, c_int64, c_int64, _P, _P, _P, _P, _P]),
    'aa_masked_mean': (c_int, [_P, c_int, c_int64, _P, c_int64, c_int32, c_int32, _P, _P, _P, _P]),
    'aa_ppo_pack_metrics': (c_int, [_P, _P, _P, _P, _P, c_int32, _P, POINTER(AaColl), _P, _P]),
    'aa_allreduce_packed': (c_int, [_P, _P, c_int32, POINTER(AaColl), _P]),
    'aa_move_padding_left': (c_int, [_P, c_int32, c_int32, c_int64, c_int64, _P, _P]),
    'aa_count_nonpad': (c_int, [_P, c_int32, c_int32, c_int64, c_int64, _P, _P]),
    'aa_ppo_rollout_layout': (c_int, [_P, c_int32, c_int64, _P, c_int32, c_int64, c_int32, c_int64, _P, _P, _P, _P]),
    'aa_tail_plan_build': (c_int, [_P, c_int32, c_int32, c_int64, c_int64, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, c_int64,
                                   c_int64, _P, _P, _P]),
    'aa_tail_rows': (c_int, [_P, c_int, c_int64, _P, c_int32, c_int32, c_int32, _P, c_int64, c_int32, _P]),
    'aa_ce_rows': (c_int, [_P, c_int32, c_int32, c_int64, c_int64, c_int64, c_int32, _P, _P, _P, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(_SIGS)


def lib() -> ctypes.CDLL:
    """Load (building first if the .so is absent and nvcc is present) libaa_b200.so."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build

        _build.build()
    try:
        handle = ctypes.CDLL(LIB_PATH)
    except OSError as e:  # loud: there is no fallback path
        raise RuntimeError(f'libaa_b200.so could not be loaded from {LIB_PATH}: {e}') from e
    for name, (res, args) in _SIGS.items():
        fn = getattr(handle, name)
        fn.restype = res
        fn.argtypes = args
    if handle.aa_abi_version() != 3:
        raise RuntimeError('libaa_b200.so ABI version mismatch: rebuild with `python -m align_anything_b200.build --force`')
    _lib = handle
    return _lib


def dtype_code(dtype: torch.dtype) -> int:
    try:
        return _DTYPE_CODE[dtype]
    except KeyError:
        raise TypeError(f'align_anything_b200: unsupported dtype {dtype} (bf16 / f16 / f32 only)') from None


def code_dtype(code: int) -> torch.dtype:
    return _CODE_DTYPE[code]


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().aa_last_error().decode(errors='replace')
        raise RuntimeError(f'libaa_b200 error {rc}: {msg}')


def ptr(t: torch.Tensor | None):
    return None if t is None else t.data_ptr()


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors: torch.Tensor) -> torch.device:
    """The product path is CUDA-only and fails loudly otherwise (no CPU fallback)."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                'align_anything_b200 runs on a B200 (sm_100a) only: got a tensor on '
                f'{t.device}.  There is deliberately no CPU fallback.'
            )
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f'tensors on different devices: {dev} vs {t.device}')
    return dev
