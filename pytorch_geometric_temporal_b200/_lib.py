"""ctypes binding of libstmp.so (the C ABI declared in include/stmp.h).

There is NO CPU fallback: importing succeeds without a GPU (so host logic can be tested), but every
compute entry point requires CUDA tensors and the library; a missing library raises immediately.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_uint32, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("STMP_LIB", os.path.join(_HERE, "lib", "libstmp.so"))   # STMP_LIB: A/B a second build of the library

STMP_OK, STMP_EINVAL, STMP_ESHAPE, STMP_EGRAPH, STMP_ECUDA, STMP_EUNSUPPORTED, STMP_ENOMEM = range(7)
FLAVOR_DCONV, FLAVOR_CHEB, FLAVOR_GCN, FLAVOR_CHEB_ATT = range(4)
NORM_NONE, NORM_SYM, NORM_RW = range(3)
GCN_IMPROVED, GCN_NO_SELF_LOOPS, DCONV_ALLOW_DUPLICATES = 1, 2, 4
NORM_CODE = {None: NORM_NONE, "sym": NORM_SYM, "rw": NORM_RW}


class StmpError(RuntimeError):
    pass


class StmpUnsupported(StmpError):
    """The fused kernel cannot take this configuration; callers route to the tiled path."""


_P = c_void_p
_SIGNATURES = {
    "stmp_plan_create": (c_int, [c_int, c_int64, c_int64, _P, _P, c_int, c_float, c_uint32, _P, POINTER(c_void_p)]),
    "stmp_plan_create_pergraph": (c_int, [c_int, c_int64, c_int64, _P, _P, c_int, _P, c_uint32, _P, POINTER(c_void_p)]),
    "stmp_plan_destroy": (None, [_P]),
    "stmp_plan_num_ops": (c_int, [_P]),
    "stmp_plan_num_nodes": (c_int64, [_P]),
    "stmp_plan_nnz": (c_int64, [_P, c_int]),
    "stmp_plan_export": (c_int, [_P, c_int, c_int, _P, _P, _P, _P, _P]),
    "stmp_spmm": (c_int, [_P, c_int, c_int, c_int64, c_int64, _P, c_int64, c_int64, _P, c_int64, c_int64, c_float,
                          _P, c_int64, c_int64, c_float, _P, _P]),
    "stmp_spmm_att_t": (c_int, [_P, c_int, c_int64, c_int64, _P, c_int64, c_int64, _P, c_int64, c_int64, c_float, _P, c_int64, c_int64,
                               c_float, _P, c_int64, _P]),
    "stmp_gemm_blocks_f32": (c_int, [c_int64, c_int64, c_int64, c_int64, _P, _P, _P, _P, c_int64, _P, _P, _P, c_int, _P, _P, c_float, _P,
                                     c_int64, _P]),
    "stmp_spatial_attention_fwd": (c_int, [c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P, c_int64, _P]),
    "stmp_astgcn_factors_fwd": (c_int, [c_int64, c_int64, c_int64, c_int64] + [_P] * 13),
    "stmp_gemm_blocks_image_bytes": (c_int64, [c_int64, c_int64]),
    "stmp_gemm_blocks_image": (c_int, [_P, c_int64, c_int64, _P, _P]),
    "stmp_spmm_att_grad": (c_int, [_P, c_int, c_int64, c_int64, _P, c_int64, c_int64, _P, c_int64, c_int64, _P, _P]),
    "stmp_dcrnn_seq_fwd": (c_int, [_P, c_int64, c_int64, c_int64, c_int64, c_int64, _P, _P, c_int64, c_int64,
                                   _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "stmp_seq_workspace_bytes": (c_int64, [_P, c_int64, c_int64]),
    "stmp_dcrnn_seq_supported": (c_int, [_P, c_int64, c_int64, c_int64]),
    "stmp_gru_seq_fwd": (c_int, [_P, c_int, c_int64, c_int64, c_int64, _P, _P, c_int64, c_int64, _P, _P, _P, c_int64, _P, _P, _P, _P, _P]),
    "stmp_gru_weight_image_bytes": (c_int64, []),
    "stmp_dcrnn_pack_weights": (c_int, [c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, _P]),
    "stmp_gru_pack_weights": (c_int, [_P, _P, _P, _P]),
    "stmp_gru_seq_supported": (c_int, [_P, c_int, c_int64, c_int64]),
    "stmp_tgcn_attn_fwd": (c_int, [_P, c_int64, c_int64, c_int64, _P, _P, c_int64, _P, _P, _P, _P, _P, _P]),
    "stmp_gru_zr": (c_int, [c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "stmp_gru_out": (c_int, [c_int64, _P, _P, _P, _P, _P, _P]),
    "stmp_dcrnn_bwd_supported": (c_int, [_P, c_int64, c_int64, c_int64]),
    "stmp_dcrnn_bwd_basis": (c_int, [_P] + [c_int64] * 4 + [_P, c_int64, c_int64, _P, _P, _P, _P, _P, c_int64, _P]),
    "stmp_dcrnn_bwd_seq": (c_int, [_P] + [c_int64] * 4 + [_P] * 11),
    "stmp_dcrnn_pack_bwd_weights": (c_int, [c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P]),
    "stmp_tgcn_attn_bwd_workspace_bytes": (c_int64, [_P, c_int64]),
    "stmp_tgcn_attn_bwd": (c_int, [_P, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "stmp_dcrnn_bwd_wgrad_workspace_bytes": (c_int64, [c_int64]),
    "stmp_dcrnn_bwd_wgrad": (c_int, [c_int64, c_int64, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "stmp_adam_flat": (c_int, [c_int64, _P, _P, _P, _P, _P, _P, c_float, c_float, c_float, c_float, c_float, c_float, c_int, _P]),
    "stmp_masked_mae_workspace_floats": (c_int64, []),
    "stmp_masked_mae_fwd": (c_int, [c_int64, _P, _P, _P, _P, _P, _P]),
    "stmp_masked_mae_bwd": (c_int, [c_int64, _P, _P, _P, _P, _P, _P]),
    "stmp_gru_bwd_carry": (c_int, [c_int64] * 5 + [_P, _P, _P, _P, _P, _P, c_int64, _P, c_int64, _P, _P, c_int64, _P, _P, _P, _P]),
    "stmp_gru_bwd_zr": (c_int, [c_int64] * 5 + [_P, _P, c_int64, _P, _P, _P, c_int64, _P, _P, _P]),
    "stmp_lstm_ifc": (c_int, [c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "stmp_lstm_gate_bwd": (c_int, [c_int64, c_int64] + [_P] * 15),
    "stmp_lstm_oh": (c_int, [c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "stmp_gemm_packed_elems": (c_int64, [c_int64, c_int64]),
    "stmp_gemm_prepack": (c_int, [_P, c_int64, c_int64, c_int64, _P, _P]),
    "stmp_gemm_f32": (c_int, [_P, c_int64, c_int64, c_int64, c_int64, _P, _P, _P, _P, c_int64, _P]),
    "stmp_gemm_lstm_f32": (c_int, [_P, c_int64, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "stmp_window_gather": (c_int, [_P, c_int64, c_int64, _P, c_int64, c_int64, _P, _P, _P]),
    "stmp_set_option": (c_int, [c_char_p, c_int]),
    "stmp_last_error": (c_char_p, []),
    "stmp_version": (c_char_p, []),
    "stmp_launch_count": (c_int64, []),
    "stmp_path_counters": (c_int, [_P, _P, c_int]),
}

_lib = None


def exported_symbols():
    return sorted(_SIGNATURES)


def lib():
    """Load (once) and return the ctypes handle.  Raises StmpError if the library is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise StmpError(
                f"{LIB_PATH} is missing: build it with `python -m pytorch_geometric_temporal_b200.build` "
                "(nvcc, sm_100a).  There is no CPU/PyTorch fallback for the hot path.")
        h = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def last_error() -> str:
    return lib().stmp_last_error().decode("utf-8", "replace")


def check(rc: int):
    if rc == STMP_OK:
        return
    msg = last_error()
    if rc == STMP_EINVAL:
        raise ValueError(msg)
    if rc == STMP_EUNSUPPORTED:
        raise StmpUnsupported(msg)
    if rc == STMP_ENOMEM:
        raise MemoryError(msg)
    raise StmpError(msg)  # ESHAPE / EGRAPH / ECUDA -> RuntimeError, like torch shape errors


def set_option(name: str, value: int):
    check(lib().stmp_set_option(name.encode(), int(value)))


def launch_count() -> int:
    return int(lib().stmp_launch_count())


def path_counters() -> dict:
    """{kernel name: launches so far} -- lets tests and users assert which path (tcgen05 / FFMA / tiled) served a call."""
    n = 96
    names = (c_char_p * n)()
    counts = (c_int64 * n)()
    k = lib().stmp_path_counters(ctypes.cast(names, c_void_p), ctypes.cast(counts, c_void_p), n)
    return {names[i].decode(): int(counts[i]) for i in range(min(k, n))}


def ptr(t):
    """Device pointer of a tensor (or None)."""
    return None if t is None else c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)
