"""ctypes binding of libpsb_b200.so (the C ABI declared in include/psb.h).

There is NO fallback: if the library is missing or a call returns a non-zero
status this module raises.  PyTorch is used only to own device memory and
streams; every op below runs hand-written sm_100a CUDA.
"""
import ctypes
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libpsb_b200.so")

c_i64, c_i32, c_f32, c_vp = ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_void_p
c_f64 = ctypes.c_double

MAX_CONTRIBS = 8
TOPK_EXACT, TOPK_TC, TOPK_TC16 = 0, 1, 2


class Contrib(ctypes.Structure):
    """psb_contrib_t (include/psb.h)."""
    _fields_ = [("idx", c_vp), ("n", c_i64), ("src", c_vp), ("src_row", c_vp), ("src_div", c_i64),
                ("scale", c_vp), ("scale2", c_vp), ("scale2_div", c_i64), ("to_bias", c_i32),
                ("reserved", c_i32)]


_ENC_NAMES = ("wq", "bq", "wk", "bk", "wv", "bv", "wo", "bo", "ln_attn_g", "ln_attn_b", "ln_ff_g", "ln_ff_b",
              "w1", "b1", "w2", "b2", "ln_out_g", "ln_out_b")


class EncoderParams(ctypes.Structure):
    """psb_encoder_params_t (also the layout of psb_encoder_grads_t)."""
    _fields_ = [(n, c_vp) for n in _ENC_NAMES]


class EncoderCfg(ctypes.Structure):
    """psb_encoder_cfg_t."""
    _fields_ = [("S", c_i64), ("T", c_i64), ("d", c_i64), ("heads", c_i64), ("ff", c_i64), ("copies", c_i64),
                ("out_pos", c_i64), ("pre_ln", c_i32), ("raw_input", c_i32), ("ln_eps", c_f32), ("p_drop", c_f32),
                ("seed_dev", c_vp), ("first", c_vp), ("table", c_vp), ("table_rows", c_i64), ("idx", c_vp),
                ("pad_idx", c_i64), ("dense", c_vp), ("mask", c_vp), ("pe", c_vp), ("first_ready", c_vp), ("wgrad_done", c_vp)]


class AdamTensor(ctypes.Structure):
    """psb_adam_tensor_t."""
    _fields_ = [("p", c_vp), ("g", c_vp), ("m", c_vp), ("v", c_vp), ("n", c_i64)]


class AdamRows(ctypes.Structure):
    """psb_adam_rows_t."""
    _fields_ = [("p", c_vp), ("m", c_vp), ("v", c_vp), ("last_step", c_vp), ("rows", c_vp), ("grad", c_vp),
                ("n_rows", c_vp), ("cap", c_i64), ("d", c_i64), ("table_rows", c_i64), ("bias_p", c_vp),
                ("bias_m", c_vp), ("bias_v", c_vp), ("bias_grad", c_vp), ("grad_by_row", c_i32), ("reserved", c_i32)]


ADAM_MAX_TENSORS = 64
ADAM_MAX_ROW_TABLES = 8
ADAM_MAX_IDX_LISTS = 8
PEER_MAX = 16
PEER_HANDLE_BYTES = 64


class FoldTable(ctypes.Structure):
    """psb_fold_table_t."""
    _fields_ = [("rows", c_vp * PEER_MAX), ("vals", c_vp * PEER_MAX), ("n_rows", c_vp * PEER_MAX), ("cap", c_i64),
                ("d", c_i64), ("shard_rows", c_i64), ("posmap", c_vp), ("dense", c_vp), ("touched", c_vp),
                ("n_touched", c_vp)]


class Corpus(ctypes.Structure):
    """psb_corpus_t."""
    _fields_ = [("review_user", c_vp), ("review_item", c_vp), ("review_uloc", c_vp), ("review_in_set", c_vp),
                ("user_seq_off", c_vp), ("user_seq", c_vp), ("item_query_off", c_vp), ("item_query", c_vp),
                ("query_words", c_vp), ("n_reviews", c_i64), ("n_users", c_i64), ("n_items", c_i64),
                ("n_queries", c_i64), ("wq", c_i64), ("word_pad", c_i64), ("item_seq_off", c_vp), ("item_seq", c_vp),
                ("review_time", c_vp)]


HIST_SEQ, HIST_LAST, HIST_RANDOM = 0, 1, 2
c_u32 = ctypes.c_uint32
c_cpp = ctypes.POINTER(ctypes.c_char_p)

# name -> (restype, argtypes); the CPU test-suite checks every symbol of psb.h is here and exported
SIGNATURES = {
    "psb_abi_version": (c_i32, []),
    "psb_status_string": (ctypes.c_char_p, [c_i32]),
    "psb_launch_count": (c_i64, []),
    "psb_profile_enable": (c_i32, [c_i32]),
    "psb_profile_dump": (c_i64, [ctypes.c_char_p, c_i64]),
    "psb_gather_rows": (c_i32, [c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "psb_gather_meanpool_fwd": (c_i32, [c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp,
                                        c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "psb_fs_bwd": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "psb_meanpool_token_weights": (c_i32, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "psb_ns_loss_fwd": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_f32,
                                c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "psb_tem_loss_fwd": (c_i32, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_f32, c_i64, c_i64, c_f32, c_vp, c_vp, c_vp,
                                 c_vp, c_vp]),
    "psb_tem_loss_finish": (c_i32, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "psb_score_rows": (c_i32, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "psb_scatter_reduce_workspace_bytes": (c_i64, [c_i64, c_i64]),
    "psb_scatter_reduce_rows": (c_i32, [ctypes.POINTER(Contrib), c_i32, c_i64, c_i64, c_i64, c_vp, c_i64,
                                        c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "psb_scatter_sort_rows": (c_i32, [ctypes.POINTER(Contrib), c_i32, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "psb_scatter_reduce_sorted": (c_i32, [ctypes.POINTER(Contrib), c_i32, c_i64, c_i64, c_i64, c_vp, c_i64,
                                          c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "psb_zero_rows": (c_i32, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "psb_catalog_topk_workspace_bytes": (c_i64, [c_i64, c_i64, c_i64, c_i64, c_i32]),
    "psb_catalog_topk": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_i32, c_vp, c_vp,
                                 c_i64, c_vp, c_vp, c_vp]),
    "psb_debug_tmem_read_bw": (c_i32, [c_i32, c_i32, c_vp]),
    "psb_debug_gemm3_tf32": (c_i32, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "psb_debug_tail_trace": (c_i32, [c_vp]),
    "psb_catalog_prepare_f16": (c_i32, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "psb_catalog_topk_f16": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64,
                                     c_vp, c_vp, c_vp]),
    "psb_table_max_row_sqnorm": (c_i32, [c_vp, c_i64, c_i64, c_vp, c_vp]),
    "psb_topk_merge": (c_i32, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "psb_adam_workspace_bytes": (c_i64, [ctypes.POINTER(AdamTensor), c_i32]),
    "psb_adam_step": (c_i32, [ctypes.POINTER(AdamTensor), c_i32, c_f64, c_f64, c_f64, c_f64, c_f64, c_f64, c_i32,
                              c_f64, c_i32, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "psb_grad_sqnorm": (c_i32, [ctypes.POINTER(AdamTensor), c_i32, c_vp, c_vp, c_i64, c_vp]),
    "psb_adam_catchup_steps": (c_i32, [c_f64, c_f64]),
    "psb_adam_sparse_workspace_bytes": (c_i64, [ctypes.POINTER(AdamTensor), c_i32, ctypes.POINTER(AdamRows), c_i32]),
    "psb_adam_sparse_step": (c_i32, [ctypes.POINTER(AdamTensor), c_i32, ctypes.POINTER(AdamRows), c_i32, c_f64, c_f64,
                                     c_f64, c_f64, c_f64, c_i32, c_f64, c_i32, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64,
                                     c_vp]),
    "psb_grad_sqnorm_sparse": (c_i32, [ctypes.POINTER(AdamTensor), c_i32, ctypes.POINTER(AdamRows), c_i32, c_vp, c_vp, c_i64,
                                       c_vp]),
    "psb_peer_gather_rows_lazy": (c_i32, [ctypes.POINTER(c_vp), ctypes.POINTER(c_vp), ctypes.POINTER(c_vp),
                                          ctypes.POINTER(c_vp), c_i32, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64,
                                          c_vp, c_f64, c_f64, c_f64, c_f64, c_i32, c_f64, c_vp, c_vp, c_i64, c_vp]),
    "psb_adam_rows_catchup": (c_i32, [ctypes.POINTER(AdamRows), ctypes.POINTER(c_vp), ctypes.POINTER(c_i64), c_i32,
                                      c_i64, c_f64, c_f64, c_f64, c_f64, c_i32, c_f64, c_vp, c_vp, c_i64, c_vp]),
    "psb_peer_alloc": (c_i32, [c_i64, ctypes.POINTER(c_vp)]),
    "psb_peer_free": (c_i32, [c_vp]),
    "psb_peer_export": (c_i32, [c_vp, ctypes.c_char_p]),
    "psb_peer_open": (c_i32, [ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    "psb_peer_close": (c_i32, [c_vp]),
    "psb_peer_barrier": (c_i32, [ctypes.POINTER(c_vp), c_i32, c_i32, c_vp, c_vp, c_i64, c_vp, c_i32, c_vp]),
    "psb_peer_gather_rows": (c_i32, [ctypes.POINTER(c_vp), c_i32, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64,
                                     c_vp, c_vp]),
    "psb_peer_fold_lists": (c_i32, [ctypes.POINTER(FoldTable), c_i32, c_i32, c_i32, c_f32, c_vp, c_vp]),
    "psb_peer_sum_sqnorm": (c_i32, [ctypes.POINTER(c_vp), c_i32, c_vp, c_vp, c_vp]),
    "psb_peer_norm_exchange": (c_i32, [ctypes.POINTER(AdamTensor), c_i32, ctypes.POINTER(AdamRows), c_i32, ctypes.POINTER(c_vp),
                                       ctypes.POINTER(c_vp), c_i32, c_i32, c_vp, c_vp, c_i64, c_vp, c_i32, c_vp, c_vp, c_vp,
                                       c_i64, c_vp]),
    "psb_peer_allreduce": (c_i32, [ctypes.POINTER(c_vp), c_i32, c_i32, c_i64, c_f32, c_vp, c_vp]),
    "psb_build_item_batch": (c_i32, [ctypes.POINTER(Corpus), c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i32, c_u32,
                                     c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "psb_build_review_test_batch": (c_i32, [ctypes.POINTER(Corpus), c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_i32,
                                            c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "psb_subset_key": (c_u32, [c_u32, c_u32, c_u32]),
    "psb_target_rank": (c_i32, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "psb_write_ranklist": (c_i64, [ctypes.c_char_p, c_cpp, c_vp, c_vp, c_cpp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i32]),
    "psb_encoder_saved_bytes": (c_i64, [ctypes.POINTER(EncoderCfg)]),
    "psb_encoder_workspace_bytes": (c_i64, [ctypes.POINTER(EncoderCfg), c_i32]),
    "psb_encoder_fwd": (c_i32, [ctypes.POINTER(EncoderCfg), ctypes.POINTER(EncoderParams), c_vp, c_i64, c_vp, c_i64,
                                c_vp, c_vp]),
    "psb_encoder_bwd": (c_i32, [ctypes.POINTER(EncoderCfg), ctypes.POINTER(EncoderParams), c_vp, c_i64, c_vp, c_i64,
                                c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(EncoderParams), c_vp]),
}

_lib = None

# Parameter-write epoch: psb_adam_step and CUDA-graph replays update parameters through raw pointers, so
# ``tensor._version`` does not change.  Every such writer bumps this counter; caches derived from parameter
# values (the fp16 shortlist copy of the item table, its row-norm bound) carry it in their key.
PARAM_EPOCH = [0]


def note_param_write():
    PARAM_EPOCH[0] += 1


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "prodsearch_b200: %s is missing -- build it with `python -m prodsearch_b200.build` "
                "(there is no CPU or PyTorch fallback for this path)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.psb_abi_version() != 1:
            raise ImportError("prodsearch_b200: ABI version mismatch in %s" % LIB_PATH)
        _lib = lib
    return _lib


def status_string(st):
    return load().psb_status_string(st).decode()


def check(st, what):
    if st != 0:
        raise RuntimeError("%s failed: status %d (%s)" % (what, st, status_string(st)))


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def ptr(t, dtype=None, allow_none=True):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        if not allow_none:
            raise ValueError("tensor required")
        return None
    if not t.is_cuda:
        raise RuntimeError("prodsearch_b200 ops need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("prodsearch_b200 ops need contiguous tensors")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError("expected dtype %s, got %s" % (dtype, t.dtype))
    return t.data_ptr()


def launch_count():
    return int(load().psb_launch_count())


def profile_enable(on=True):
    """Bracket every kernel the library launches (outside graph capture) with CUDA events."""
    check(load().psb_profile_enable(1 if on else 0), "psb_profile_enable")


def profile_dump():
    """{kernel name: (launches, total_ms, min_ms, max_ms)} since profile_enable / the last dump (synchronises)."""
    buf = ctypes.create_string_buffer(1 << 16)
    n = load().psb_profile_dump(buf, len(buf))
    if n < 0:
        raise RuntimeError("psb_profile_dump failed: %d" % n)
    out = {}
    for line in buf.value.decode().splitlines():
        name, cnt, tot, mn, mx = line.split()
        out[name] = (int(cnt), float(tot), float(mn), float(mx))
    return out
