"""ctypes binding of librsa_b200.so (C ABI declared in include/rsa.h).

There is no CPU fallback: importing this module without the built library raises, and every call that touches
the GPU raises RsaError when the library reports a failure."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librsa_b200.so")

RSA_OK = 0
FAMILY_WAN, FAMILY_JOINT = 0, 1
MASK_BUILD, MASK_KEEP_LISTS, MASK_KEEP_ALL = 0, 1, 2   # enum rsa_mask_mode
DTYPE_BF16, DTYPE_F16 = 0, 1                           # enum rsa_dtype
ATTN_FP32_SCALE = 256                                  # RSA_ATTN_FP32_SCALE, OR-ed into rsa_masked_attention's dtype
BLOCK = 128


class RsaError(RuntimeError):
    pass


class AttnDesc(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("heads", C.c_int32), ("seq", C.c_int32), ("head_dim", C.c_int32),
        ("q_stride", C.c_int64 * 3), ("k_stride", C.c_int64 * 3), ("v_stride", C.c_int64 * 3),
        ("o_stride", C.c_int64 * 3),
        ("family", C.c_int32), ("n_blocks", C.c_int32), ("nq_blocks", C.c_int32), ("text_keys", C.c_int32),
        ("kv_len", C.c_int32), ("kv_zero_from", C.c_int32), ("text_end_block", C.c_int32),
        ("text_q_valid", C.c_int32), ("top_k", C.c_int32), ("p_remain", C.c_float),
        ("first_frame_blocks", C.c_int32), ("nbr_rows", C.c_int32), ("nbr_cols", C.c_int32),
        ("nbr", C.c_void_p), ("debug_dump_probs", C.c_int32), ("vis_len", C.c_int32), ("dtype", C.c_int32),
    ]


class WsView(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "q_pool", "q_mad", "k_cat", "k_mad", "v_pool", "scores", "nogapr", "probs", "w_skip", "mask_bits",
        "kept_idx", "kept_cnt", "n_needed", "R", "C")] + [(n, C.c_int32) for n in (
            "nkc", "score_ld", "n_entries", "ent_ld", "mask_words", "nqt", "nogapr_ld", "reserved")] + [
                ("sched_idx", C.c_void_p), ("pair_shared", C.c_void_p), ("quad_shared", C.c_void_p)]


class PrepDesc(C.Structure):
    _fields_ = [("rows", C.c_int32), ("dst_row", C.c_int32), ("src_stride", (C.c_int64 * 2) * 3),
                ("norm", C.c_int32), ("eps", C.c_float), ("q_weight", C.c_void_p), ("k_weight", C.c_void_p),
                ("rope_rows", C.c_int32), ("rope_compact", C.c_int32), ("cos", C.c_void_p), ("sin", C.c_void_p),
                ("row_scratch", C.c_void_p), ("q_bias", C.c_void_p), ("k_bias", C.c_void_p)]


class PeerRoute(C.Structure):
    _fields_ = [("n_ranks", C.c_int32), ("rank", C.c_int32), ("rows_per_rank", C.c_int32), ("heads_total", C.c_int32),
                ("head0", C.c_int32), ("reserved", C.c_int32), ("src_table", C.c_void_p), ("src_stride", C.c_int64 * 2), ("out_table", C.c_void_p),
                ("out_stride", C.c_int64 * 2), ("rinv_table", C.c_void_p)]


EXPORTS = [
    "rsa_last_error_string", "rsa_version", "rsa_device_ok", "rsa_gilbert_map", "rsa_gilbert_block_neighbors",
    "rsa_permute_rows", "rsa_attn_workspace_bytes", "rsa_attn_workspace_view", "rsa_pool_stats",
    "rsa_block_scores", "rsa_block_select", "rsa_rect_c", "rsa_sparse_attention", "rsa_rectified_attention",
    "rsa_masked_attention_workspace_bytes", "rsa_masked_attention",
    "rsa_debug_set_attention_dump", "rsa_debug_set_attention_flags", "rsa_host_call_scratch_bytes",
    "rsa_rectified_attention_host", "rsa_qkv_prep", "rsa_rectified_attention_pooled", "rsa_peer_alloc",
    "rsa_peer_free", "rsa_peer_export", "rsa_peer_open", "rsa_peer_close", "rsa_qkv_prep_gather",
    "rsa_rectified_attention_pooled_scatter", "rsa_rectified_attention_reuse",
    "rsa_debug_attention_grid_slot", "rsa_debug_front_text_heads", "rsa_gilbert_xyz2d_r",
    "rsa_attn_desc_size", "rsa_prep_desc_size", "rsa_peer_route_size", "rsa_row_rms",
    "rsa_dense_attention", "rsa_dense_attention_scatter", "rsa_row_rms_dtype",
]

_lib = None


ABI_VERSION = 110


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RsaError(
            f"{LIB_PATH} is missing: build it with `python rectified-spaattn_b200/build_native.py` "
            "(there is no CPU or PyTorch fallback for this path)")
    L = C.CDLL(LIB_PATH)
    p, i32, i64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
    L.rsa_last_error_string.restype = C.c_char_p
    L.rsa_version.restype = i32
    if L.rsa_version() != ABI_VERSION:   # the ctypes structures below mirror include/rsa.h of exactly this version
        raise RsaError(f"{LIB_PATH} has ABI version {L.rsa_version()}, this package expects {ABI_VERSION}: rebuild it "
                       "with `python rectified-spaattn_b200/build_native.py`")
    L.rsa_device_ok.restype = i32
    for n in ("rsa_attn_desc_size", "rsa_prep_desc_size", "rsa_peer_route_size"):
        getattr(L, n).restype = sz
    if (L.rsa_attn_desc_size(), L.rsa_prep_desc_size(), L.rsa_peer_route_size()) != (
            C.sizeof(AttnDesc), C.sizeof(PrepDesc), C.sizeof(PeerRoute)):
        raise RsaError("ctypes structures of rsa_b200/native.py do not match the library's include/rsa.h")
    L.rsa_gilbert_map.argtypes = [i32, i32, i32, C.c_char_p, p, p]
    L.rsa_gilbert_block_neighbors.argtypes = [i32, i32, i32, i32, C.c_char_p, p]
    L.rsa_gilbert_xyz2d_r.argtypes = [i64] * 16
    L.rsa_gilbert_xyz2d_r.restype = i64
    L.rsa_permute_rows.argtypes = [p, p, p, i32, i64, i64, i64, i64, i64, p]
    L.rsa_attn_workspace_bytes.argtypes = [C.POINTER(AttnDesc)]
    L.rsa_attn_workspace_bytes.restype = sz
    L.rsa_attn_workspace_view.argtypes = [C.POINTER(AttnDesc), p, sz, C.POINTER(WsView)]
    L.rsa_pool_stats.argtypes = [C.POINTER(AttnDesc), p, p, p, p, sz, p]
    for n in ("rsa_block_scores", "rsa_block_select", "rsa_rect_c"):
        getattr(L, n).argtypes = [C.POINTER(AttnDesc), p, sz, p]
    L.rsa_sparse_attention.argtypes = [C.POINTER(AttnDesc), p, p, p, p, p, sz, p]
    L.rsa_rectified_attention.argtypes = [C.POINTER(AttnDesc), p, p, p, p, p, sz, p]
    L.rsa_masked_attention_workspace_bytes.argtypes = [i32, i32, i32]
    L.rsa_masked_attention_workspace_bytes.restype = sz
    L.rsa_masked_attention.argtypes = [p, p, p, p, i32, i32, i32, i32, C.POINTER(i64), C.POINTER(i64),
                                       C.POINTER(i64), C.POINTER(i64), p, i32, i32, p, sz, p, i32, i32]
    L.rsa_host_call_scratch_bytes.argtypes = [C.POINTER(AttnDesc), i32]
    L.rsa_host_call_scratch_bytes.restype = sz
    L.rsa_rectified_attention_host.argtypes = [C.POINTER(AttnDesc), p, p, p, p, i32, p, sz, p]
    L.rsa_qkv_prep.argtypes = [C.POINTER(PrepDesc), C.POINTER(AttnDesc), p, p, p, p, p, p, i32, p, sz, p]
    L.rsa_rectified_attention_pooled.argtypes = [C.POINTER(AttnDesc), p, p, p, p, p, sz, p]
    L.rsa_rectified_attention_reuse.argtypes = [C.POINTER(AttnDesc), p, p, p, p, p, sz, i32, i32, p]
    L.rsa_qkv_prep_gather.argtypes = [C.POINTER(PrepDesc), C.POINTER(AttnDesc), C.POINTER(PeerRoute), p, p, p, i32, p,
                                      sz, p]
    L.rsa_rectified_attention_pooled_scatter.argtypes = [C.POINTER(AttnDesc), p, p, p, C.POINTER(PeerRoute), p, sz, p]
    L.rsa_dense_attention.argtypes = [C.POINTER(AttnDesc), p, p, p, p, i32, i32, i32, p]
    L.rsa_dense_attention_scatter.argtypes = [C.POINTER(AttnDesc), p, p, p, C.POINTER(PeerRoute), i32, i32, p]
    L.rsa_row_rms.argtypes = [p, p, i32, i32, i32, C.POINTER(i64), C.POINTER(i64), C.c_float, p, p, p]
    L.rsa_row_rms_dtype.argtypes = [p, p, i32, i32, i32, C.POINTER(i64), C.POINTER(i64), C.c_float, p, p, i32, p]
    L.rsa_peer_alloc.argtypes = [sz, C.POINTER(p)]
    L.rsa_peer_free.argtypes = [p]
    L.rsa_peer_export.argtypes = [p, p]
    L.rsa_peer_open.argtypes = [p, C.POINTER(p)]
    L.rsa_peer_close.argtypes = [p]
    L.rsa_debug_set_attention_dump.argtypes = [p]
    L.rsa_debug_set_attention_dump.restype = None
    L.rsa_debug_set_attention_flags.argtypes = [i32]
    L.rsa_debug_set_attention_flags.restype = None
    L.rsa_debug_attention_grid_slot.argtypes = [i32, i32, i32, i32, i32, i32, C.POINTER(C.c_int * 5)]
    L.rsa_debug_attention_grid_slot.restype = None
    L.rsa_debug_front_text_heads.argtypes = [C.POINTER(AttnDesc)]
    L.rsa_debug_front_text_heads.restype = i32
    for n in EXPORTS:
        getattr(L, n)            # every symbol of include/rsa.h must be there
    _lib = L
    return L


def check(rc, what):
    if rc != RSA_OK:
        raise RsaError(f"{what} failed ({rc}): {lib().rsa_last_error_string().decode()}")
