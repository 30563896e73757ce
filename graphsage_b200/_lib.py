"""ctypes binding of libgraphsage_b200.so (the C-ABI in include/graphsage_b200.h).

There is deliberately no CPU fallback: if the library is missing, or a compute entry is
called without a CUDA device, the call raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libgraphsage_b200.so")

ABI_VERSION = 2          # GS_ABI_VERSION of include/graphsage_b200.h this binding was written against
GS_F32, GS_BF16 = 0, 1
ACT_NONE, ACT_RELU = 0, 1
COMBINE_ADD, COMBINE_CONCAT = 0, 1
MATH_FP32_SIMT, MATH_TF32X3, MATH_TF32, MATH_BF16 = 0, 1, 2, 3
MAX_SEGMENTS = 4

c_i32, c_i64, c_u64, c_vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64, ctypes.c_void_p


class Segment(ctypes.Structure):
    _fields_ = [("self_ids", c_vp), ("neigh_ids", c_vp), ("self_row0", c_i64), ("neigh_row0", c_i64),
                ("n", c_i64), ("k", c_i32), ("_pad", c_i32), ("out_row0", c_i64)]


MAX_SHARDS = 16


class ShardedTable(ctypes.Structure):
    _fields_ = [("base", c_vp * MAX_SHARDS), ("row_start", c_i64 * (MAX_SHARDS + 1)), ("n_shards", c_i32),
                ("my_shard", c_i32), ("n_global_rows", c_i64), ("zero_row", c_i64), ("remap", c_vp)]


class GemmPart(ctypes.Structure):
    _fields_ = [("A", c_vp), ("lda", c_i64), ("K", c_i32), ("B", c_vp), ("ldb", c_i64), ("N", c_i32)]


_SIGNATURES = {
    "gs_version": (c_i32, []),
    "gs_last_error_string": (ctypes.c_char_p, []),
    "gs_set_tuning": (c_i32, [ctypes.c_char_p, c_i32]),
    "gs_sample_padded": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_vp, c_u64, c_u64, c_vp, c_vp, c_vp]),
    "gs_sample_padded_khop": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_i64, ctypes.POINTER(c_i32), c_i32, c_u64, c_u64, c_vp,
                                      ctypes.POINTER(c_vp), c_vp]),
    "gs_build_padded_adj": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_u64, c_u64, c_vp, c_vp, c_vp]),
    "gs_sample_unigram": (c_i32, [c_vp, c_i64, c_i32, c_u64, c_u64, c_vp, c_vp, c_vp]),
    "gs_sample_csr": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i64, c_i32, c_i32, c_u64, c_u64, c_vp, c_i32, c_vp, c_vp]),
    "gs_perm_prefix_host": (c_i32, [c_u64, c_u64, c_i32, c_i32, ctypes.POINTER(c_i32)]),
    "gs_gather_rows": (c_i32, [c_vp, c_i32, c_i64, c_i32, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "gs_gather_mean": (c_i32, [c_vp, c_i32, c_i64, c_i32, c_i64, ctypes.POINTER(Segment), c_i32, c_i32, c_vp, c_vp,
                               c_i64, c_vp]),
    "gs_gather_mean_sharded": (c_i32, [ctypes.POINTER(ShardedTable), c_i32, c_i32, c_i64, ctypes.POINTER(Segment), c_i32,
                                       c_i32, c_i32, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gs_halo_begin": (c_i32, [c_vp, c_i64, c_vp, c_vp]),
    "gs_halo_claim": (c_i32, [ctypes.POINTER(ShardedTable), c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gs_halo_fetch": (c_i32, [ctypes.POINTER(ShardedTable), c_i32, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "gs_halo_translate": (c_i32, [ctypes.POINTER(ShardedTable), c_vp, c_i64, c_vp, c_vp, c_vp]),
    "gs_translate_ids": (c_i32, [ctypes.POINTER(ShardedTable), c_vp, c_i64, c_vp, c_vp]),
    "gs_gather_rows_sharded": (c_i32, [ctypes.POINTER(ShardedTable), c_i32, c_i32, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "gs_shard_alloc": (c_i32, [c_i64, ctypes.POINTER(c_vp)]),
    "gs_shard_free": (c_i32, [c_vp]),
    "gs_ipc_export": (c_i32, [c_vp, ctypes.c_char_p]),
    "gs_ipc_import": (c_i32, [ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    "gs_ipc_close": (c_i32, [c_vp]),
    "gs_gather_rows_f32": (c_i32, [c_vp, c_i32, c_i64, c_i32, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp]),
    "gs_cast_rows_bf16": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_i64, c_vp]),
    "gs_rmat_degrees": (c_i32, [c_i32, c_i64, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                ctypes.c_double, c_u64, c_u64, c_u64, c_u64, c_vp, c_vp]),
    "gs_rmat_fill": (c_i32, [c_i32, c_i64, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, c_u64, c_u64,
                             c_u64, c_u64, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "gs_segment_max": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_i64, c_vp, c_i64, c_vp]),
    "gs_sage_gemm_workspace_bytes": (c_i64, [c_i64, ctypes.POINTER(GemmPart), c_i32, c_i32]),
    "gs_sage_gemm": (c_i32, [c_i64, ctypes.POINTER(GemmPart), c_i32, c_i32, c_vp, c_i32, c_i32, c_vp, c_i64, c_vp,
                             c_vp]),
    "gs_sage_gemm_pack": (c_i32, [ctypes.POINTER(GemmPart), c_i32, c_i32, c_vp, c_vp]),
    "gs_sage_gemm_prepacked": (c_i32, [c_i64, ctypes.POINTER(GemmPart), c_i32, c_i32, c_vp, c_i32, c_i32, c_vp, c_i64,
                                       c_vp, c_vp]),
    "gs_gather_mean_img_bytes": (c_i64, [c_i64, c_i32, c_i32]),
    "gs_gather_mean_img": (c_i32, [c_vp, c_i64, ctypes.POINTER(ShardedTable), c_i32, c_vp, c_i32, c_i64, ctypes.POINTER(Segment),
                                   c_i32, c_i32, c_i32, c_vp, c_vp]),
    "gs_sage_gemm_img": (c_i32, [c_i64, ctypes.POINTER(GemmPart), c_i32, c_i32, c_vp, c_i32, c_vp, c_i64, c_vp, c_vp, c_i32,
                                 c_vp]),
    "gs_sage_layer_small": (c_i32, [c_vp, c_i64, c_i32, c_i64, ctypes.POINTER(Segment), c_i32, ctypes.POINTER(GemmPart),
                                    c_i32, c_i32, c_vp, c_i32, c_i32, c_vp, c_i64, c_vp, c_u64, c_vp]),
    "gs_maxpool_mlp_workspace_bytes": (c_i64, [c_i32, c_i32]),
    "gs_maxpool_mlp_pack": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    "gs_maxpool_mlp_fused": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_i32, c_vp, c_i64,
                                     c_vp]),
    "gs_meanpool_mlp_fused": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_i32, c_vp, c_i64,
                                      c_vp]),
    "gs_pipeline_step": (c_i32, [c_vp, c_vp, c_i64, ctypes.POINTER(c_vp), c_i32, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp,
                                 c_vp, c_vp]),
    "gs_row_used": (c_i32, [c_vp, c_i32, c_i64, c_i32, c_i64, c_vp, c_vp]),
    "gs_lstm_seq": (c_i32, [c_vp, c_i64, c_vp, c_i32, c_vp, c_vp, c_i64, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "gs_l2_normalize_rows": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp]),
    "gs_bump_counter": (c_i32, [c_vp, c_u64, c_vp]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "graphsage_b200: %s is missing - build it with `python -m graphsage_b200.build` "
                "(there is no CPU fallback)" % LIB_PATH)
        _lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(_lib, name)          # AttributeError = symbol not exported
            fn.restype, fn.argtypes = res, args
        if _lib.gs_version() != ABI_VERSION:
            raise ImportError("graphsage_b200: %s has ABI version %d, this binding needs %d - rebuild it"
                              % (LIB_PATH, _lib.gs_version(), ABI_VERSION))
        for kv in os.environ.get("GS_TUNING", "").split(","):      # e.g. GS_TUNING=gather_variant=2,gather_ctas_per_sm=3
            if "=" in kv:
                k, v = kv.split("=", 1)
                _lib.gs_set_tuning(k.strip().encode(), int(v))
    return _lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(rc):
    if rc != 0:
        msg = lib().gs_last_error_string().decode("utf-8", "replace")
        raise RuntimeError("libgraphsage_b200 error %d: %s" % (rc, msg))


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return 0 if t is None else t.data_ptr()


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("graphsage_b200: tensor on %s - the hot path is CUDA-only (no CPU fallback)" % t.device)


def set_tuning(key, value):
    return lib().gs_set_tuning(key.encode(), int(value))


def perm_prefix_host(seed, counter, max_deg, k):
    buf = (c_i32 * max(k, 1))()
    check(lib().gs_perm_prefix_host(seed & (2**64 - 1), counter & (2**64 - 1), max_deg, k, buf))
    return list(buf[:k])
