"""ctypes binding of include/ge2e_b200.h.  There is no fallback: a missing library raises."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

_f32p = C.c_void_p   # device pointers travel as integers (tensor.data_ptr())
_i32p = C.c_void_p
_stream = C.c_void_p

SOFTMAX, CONTRAST = 0, 1
FP32, TF32, FP32_SPLIT, F16 = 0, 1, 2, 3
VARIANTS = {"softmax": SOFTMAX, "contrast": CONTRAST}
# "fp32" (the default, the reference's arithmetic) means fp32-class results: on the tensor cores through the
# split-fp16 operand mode where the shape is covered (resolve_precision), else the SIMT fp32 FMA kernels.
# "fp32_simt" / "fp32_split" pin one of the two.
# "f16": the 2e-3 tolerance class with fp16 operands instead of TF32 (same 11-bit mantissa, twice the MMA rate:
# GE2E_F16).  Opt-in: it wins only where the MMAs dominate (config 4 on one GPU: 1.12x, DESIGN 3.4).
PRECISIONS = {"fp32": FP32, "tf32": TF32, "fp32_simt": FP32, "fp32_split": FP32_SPLIT, "tf32_mma": TF32, "f16": F16}
# element type of E / dE (enum ge2e_dtype): only these two tensors may be bf16 / fp16, every other buffer is fp32
DT_F32, DT_BF16, DT_F16 = 0, 1, 2


def resolve_precision(name: str, n_local: int, n_total: int, M: int, D: int, variant: int) -> int:
    """Precision code handed to the C ABI for a (shape, variant): "fp32" picks GE2E_FP32_SPLIT where
    ge2e_b200_path() covers it (speaker shards included: a centroid row carries both of its planes)."""
    if name not in PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
    if name == "fp32" and lib().ge2e_b200_path(n_local, n_total, M, D, variant, FP32_SPLIT) == 2:
        return FP32_SPLIT
    if name == "f16" and lib().ge2e_b200_path(n_local, n_total, M, D, variant, F16) != 3:
        return TF32           # shapes the fp16-operand kernels do not cover: the TF32 permission
    return PRECISIONS[name]


def prepares_dE_hat(n_local: int, n_total: int, M: int, D: int, variant: int, precision: int) -> bool:
    """True where the softmax loss runs on tensor cores: there a forward with a backward to follow also leaves the
    un-normalised dE_hat rows + row_scale (ge2e_b200_fwd_rows), the backward rows stage is the centroid pass alone,
    and the finalize applies row_scale."""
    return variant == SOFTMAX and lib().ge2e_b200_path(n_local, n_total, M, D, variant, precision) > 0

def check_backward_shape(M: int, D: int) -> None:
    """ValueError (before anything is launched) for an M whose backward the kernels cannot run at width D."""
    m = lib().ge2e_b200_max_utterances(D)
    if M > m:
        raise ValueError(f"the GE2E backward supports at most {m} utterances per speaker at D = {D} (got M = {M}); "
                         "its last stage keeps a speaker's 2 M + 2 rows in 200 KB of shared memory")


def planes_need_copy(ptr: int, precision: int, element_size: int = 4) -> bool:
    """The fp16-plane precisions read E four elements at a time (16 bytes for fp32, 8 for bf16 / fp16): an E at
    another offset of its allocation is copied."""
    return precision in (FP32_SPLIT, F16) and ptr % (4 * element_size) != 0

# name -> (restype, argtypes); kept in the order of include/ge2e_b200.h
PROTOTYPES = {
    "ge2e_b200_version": (C.c_int, []),
    "ge2e_b200_strerror": (C.c_char_p, [C.c_int]),
    "ge2e_b200_last_cuda_error": (C.c_int, []),
    "ge2e_b200_launch_count": (C.c_ulonglong, []),
    "ge2e_b200_path": (C.c_int, [C.c_int] * 6),
    "ge2e_b200_max_utterances": (C.c_int, [C.c_int]),
    "ge2e_b200_debug_trace": (None, [C.c_void_p, C.c_int]),
    "ge2e_b200_debug_stamps": (None, [C.c_void_p]),
    "ge2e_b200_debug_hybrid": (None, [C.c_int]),
    "ge2e_b200_debug_step_schedule": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p]),
    "ge2e_b200_debug_step_model": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ge2e_b200_check_device": (C.c_int, []),
    "ge2e_b200_workspace_bytes": (C.c_size_t, [C.c_int] * 6),
    "ge2e_b200_prep": (C.c_int, [_f32p, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, _f32p, _f32p, _f32p,
                                 _stream]),
    "ge2e_b200_fwd_rows": (C.c_int, [_f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     _f32p, _f32p, C.c_float, C.c_int, C.c_int, _f32p, _i32p, _f32p, _f32p,
                                     _f32p, _f32p, _f32p, _f32p, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_bwd_rows": (C.c_int, [_f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int, C.c_int,
                                     _f32p, _f32p, _f32p, _f32p, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_bwd_finalize": (C.c_int, [_f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int,
                                         _f32p, _f32p, C.c_float, C.c_int, _f32p, _f32p, _stream]),
    "ge2e_b200_step_rows": (C.c_int, [_f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, _f32p,
                                      C.c_float, C.c_int, C.c_int, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p, _f32p,
                                      _f32p, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_peer_publish": (C.c_int, [_f32p, C.c_void_p, C.c_int, C.c_int, C.c_longlong, _f32p, C.c_longlong,
                                         _stream]),
    "ge2e_b200_step_rows_peers": (C.c_int, [_f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p,
                                            _f32p, C.c_float, C.c_int, C.c_int, _f32p, _f32p, _i32p, _f32p, _f32p,
                                            _f32p, _f32p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_forward": (C.c_int, [_f32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int,
                                    C.c_int, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p, _f32p, C.c_void_p,
                                    C.c_size_t, _stream]),
    "ge2e_b200_backward": (C.c_int, [_f32p, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, C.c_int, C.c_int,
                                     C.c_int, _f32p, _f32p, C.c_float, C.c_int, C.c_int, _f32p, _f32p,
                                     _f32p, _f32p, _f32p, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_prep_indexed": (C.c_int, [_f32p, _i32p, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, _f32p, _f32p,
                                         _f32p, _stream]),
    "ge2e_b200_bwd_finalize_indexed": (C.c_int, [_f32p, _i32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_int,
                                                 C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int, _f32p, _f32p,
                                                 _stream]),
    "ge2e_b200_forward_indexed": (C.c_int, [_f32p, _i32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int,
                                            C.c_int, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p, _f32p,
                                            C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_backward_indexed": (C.c_int, [_f32p, _i32p, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, C.c_int,
                                             C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int, C.c_int, _f32p, _f32p,
                                             _f32p, _f32p, _f32p, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_scale_bias_sgd": (C.c_int, [_f32p, _f32p, _f32p, _f32p, C.c_float, C.c_float, _f32p, _stream]),
    "ge2e_b200_debug_small_step": (None, [C.c_int]),
    "ge2e_b200_step_workspace_bytes": (C.c_size_t, [C.c_int] * 5),
    "ge2e_b200_step_launches": (C.c_int, [C.c_int] * 5),
    "ge2e_b200_scale_grads": (C.c_int, [_f32p, _f32p, C.c_longlong, _f32p, _f32p, _f32p, _stream]),
    "ge2e_b200_scale_grads_typed": (C.c_int, [_f32p, C.c_void_p, C.c_int, C.c_longlong, _f32p, _f32p, _f32p, _stream]),
    "ge2e_b200_forward_backward": (C.c_int, [_f32p, _i32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int,
                                             C.c_int, _f32p, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p,
                                             _f32p, _f32p, _f32p, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_gather_spans": (C.c_int, [_f32p, C.c_void_p, C.c_int, C.c_longlong, C.c_int, _f32p, _stream]),
    "ge2e_b200_embed_tail_fwd": (C.c_int, [_f32p, C.c_longlong, _f32p, _f32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p,
                                           _stream]),
    "ge2e_b200_embed_tail_bwd_rows": (C.c_int, [_f32p, _f32p, _f32p, C.c_int, C.c_int, _f32p, _f32p, _stream]),
    "ge2e_b200_embed_tail_bwd_gemms_supported": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong]),
    "ge2e_b200_embed_tail_bwd_gemms": (C.c_int, [_f32p, _f32p, _f32p, C.c_longlong, C.c_int, C.c_int, C.c_int,
                                                 _f32p, C.c_longlong, _f32p, _stream]),
    "ge2e_b200_threshold_counts_scratch_bytes": (C.c_size_t, [C.c_int]),
    "ge2e_b200_threshold_counts": (C.c_int, [_f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_prep_typed": (C.c_int, [C.c_void_p, C.c_int, _i32p, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, _f32p,
                                       _f32p, _f32p, _stream]),
    "ge2e_b200_bwd_finalize_typed": (C.c_int, [C.c_void_p, C.c_int, _i32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p,
                                               C.c_int, C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int, _f32p,
                                               C.c_void_p, C.c_int, _stream]),
    "ge2e_b200_forward_typed": (C.c_int, [C.c_void_p, C.c_int, _i32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p,
                                          C.c_float, C.c_int, C.c_int, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p,
                                          _f32p, _f32p, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_backward_typed": (C.c_int, [C.c_void_p, C.c_int, _i32p, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p,
                                           C.c_int, C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int, C.c_int, _f32p,
                                           _f32p, _f32p, _f32p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_forward_backward_typed": (C.c_int, [C.c_void_p, C.c_int, _i32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p,
                                                   C.c_float, C.c_int, C.c_int, _f32p, _f32p, _f32p, _f32p, _f32p,
                                                   _i32p, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_void_p, C.c_int,
                                                   C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_forward_per_row_typed": (C.c_int, [C.c_void_p, C.c_int, _i32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p,
                                                  C.c_float, C.c_int, C.c_int, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p,
                                                  _f32p, _f32p, _f32p, _f32p, C.c_void_p, C.c_size_t, _stream]),
    "ge2e_b200_backward_per_row_typed": (C.c_int, [C.c_void_p, C.c_int, _i32p, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p,
                                                   _f32p, C.c_int, C.c_int, C.c_int, _f32p, _f32p, C.c_float, C.c_int,
                                                   C.c_int, _f32p, _f32p, _f32p, _f32p, C.c_void_p, C.c_int, C.c_void_p,
                                                   C.c_size_t, _stream]),
    "ge2e_b200_centroids": (C.c_int, [_f32p, C.c_int, C.c_int, C.c_int, _f32p, _stream]),
    "ge2e_b200_utterance_centroids": (C.c_int, [_f32p, C.c_int, C.c_int, C.c_int, _f32p, _stream]),
    "ge2e_b200_normalize_rows": (C.c_int, [_f32p, C.c_int, C.c_int, _f32p, _stream]),
    "ge2e_b200_calc_loss": (C.c_int, [_f32p, C.c_int, C.c_int, C.c_float, C.c_int, _f32p, _f32p,
                                      _stream]),
}

_lib = None


class GE2ELibraryError(RuntimeError):
    pass


def lib():
    """Load csrc/libge2e_b200.so once.  Raises if it has not been built (no CPU fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GE2ELibraryError(
                f"{LIB_PATH} is missing: build it with `python -m speaker_embedding_ge2e_loss_b200.build` "
                "(needs nvcc; sm_100a only).  This package has no CPU / PyTorch fallback.")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(h, name)   # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        h = lib()
        msg = h.ge2e_b200_strerror(rc).decode()
        if rc == -6:
            msg += f" [cudaError={h.ge2e_b200_last_cuda_error()}]"
        exc = ValueError if rc in (-1, -3) else RuntimeError
        raise exc(f"{what}: {msg}")
