"""ctypes binding of include/samd_b200.h (libsamd_b200.so).

There is no CPU fallback: if the library is missing, or a compute entry point is called
without a CUDA device, this module raises.  Build the library with
`python __graft_entry__.py build` (or `make -C sam-decoding_b200/csrc`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsamd_b200.so")

FLAVOUR_SAMD = 0
FLAVOUR_SAM_ONLY = 1
DRAFT_DYN_SEQ = 0
DRAFT_STATIC_SEQ = 1
DRAFT_TREE_MODEL = 2
DRAFT_STATIC_TREE = 3
DTYPE_BF16 = 0
DTYPE_FP16 = 1
DTYPE_FP32 = 2
STOP_MAX_SEQS = 16
STOP_MAX_LEN = 16
BIAS_MAX = 256
BAD_MAX_SEQS = 16
BAD_MAX_LEN = 16

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u8p = C.POINTER(C.c_uint8)
vp = C.c_void_p


class StepArgs(C.Structure):
    _fields_ = [
        ("dyn", vp), ("stat", vp), ("static_cursor_dev", vp), ("tokens_dev", vp), ("token_stride", C.c_int32),
        ("counts_dev", vp), ("start_tok_dev", vp), ("flavour", C.c_int32), ("n_predicts", C.c_int32),
        ("len_bias", C.c_int32), ("len_threshold", C.c_int32), ("alpha", C.c_double),
        ("out_type_dev", vp), ("out_match_dyn_dev", vp), ("out_match_static_dev", vp), ("out_index_dyn_dev", vp),
        ("out_index_static_dev", vp), ("out_draft_dev", vp), ("draft_stride", C.c_int32), ("out_draft_len_dev", vp),
    ]


class VerifyArgs(C.Structure):
    _fields_ = [
        ("logits_dev", vp), ("dtype", C.c_int32), ("batch", C.c_int32), ("n_nodes", C.c_int32), ("vocab", C.c_int32),
        ("batch_stride", C.c_int64), ("row_stride", C.c_int64), ("tree_tokens_dev", vp), ("n_nodes_dev", vp),
        ("retrieve_dev", vp), ("n_paths", C.c_int32), ("depth", C.c_int32), ("retrieve_batch_stride", C.c_int64),
        ("n_paths_dev", vp), ("kv_ptrs_dev", vp), ("n_kv", C.c_int32), ("n_heads", C.c_int32), ("row_bytes", C.c_int32),
        ("kv_batch_stride", C.c_int64), ("kv_head_stride", C.c_int64), ("kv_pos_stride", C.c_int64),
        ("move_kv", C.c_int32), ("cache_len_dev", vp), ("out_best_dev", vp), ("out_accept_len_dev", vp),
        ("out_next_token_dev", vp), ("out_tokens_dev", vp), ("out_indices_dev", vp), ("out_node_argmax_dev", vp),
        ("out_topk_dev", vp), ("recycle_table_dev", vp), ("recycle_owner_dev", vp),
    ]


class SampleArgs(C.Structure):
    _fields_ = [
        ("logits_dev", vp), ("dtype", C.c_int32), ("batch", C.c_int32), ("n_nodes", C.c_int32), ("vocab", C.c_int32),
        ("batch_stride", C.c_int64), ("row_stride", C.c_int64), ("tree_tokens_dev", vp), ("retrieve_dev", vp),
        ("n_paths", C.c_int32), ("depth", C.c_int32), ("retrieve_batch_stride", C.c_int64), ("n_paths_dev", vp),
        ("temperature", C.c_float), ("top_p", C.c_float), ("top_k", C.c_int32), ("seeds_dev", vp), ("offsets_dev", vp),
        ("out_best_dev", vp), ("out_accept_len_dev", vp), ("out_next_token_dev", vp), ("out_tokens_dev", vp),
        ("out_indices_dev", vp), ("out_sample_p_dev", vp),
    ]


class SampleRequestArgs(C.Structure):
    _fields_ = [
        ("temperature_dev", vp), ("top_p_dev", vp), ("top_k_dev", vp), ("greedy_dev", vp), ("done_dev", vp),
        ("n_nodes_dev", vp), ("depth_dev", vp),
    ]


class LogprobArgs(C.Structure):
    _fields_ = [
        ("logits_dev", vp), ("dtype", C.c_int32), ("batch", C.c_int32), ("n_nodes", C.c_int32), ("vocab", C.c_int32),
        ("batch_stride", C.c_int64), ("row_stride", C.c_int64), ("indices_dev", vp), ("width", C.c_int32),
        ("count_dev", vp), ("tokens_dev", vp), ("next_token_dev", vp), ("n_nodes_dev", vp), ("done_dev", vp),
        ("n_top", C.c_int32), ("out_logprob_dev", vp), ("out_next_logprob_dev", vp), ("out_top_ids_dev", vp),
        ("out_top_logprob_dev", vp), ("out_next_top_ids_dev", vp), ("out_next_top_logprob_dev", vp),
    ]


class PenaltyArgs(C.Structure):
    _fields_ = [
        ("logits_dev", vp), ("dtype", C.c_int32), ("batch", C.c_int32), ("n_nodes", C.c_int32), ("vocab", C.c_int32),
        ("batch_stride", C.c_int64), ("row_stride", C.c_int64), ("tokens_dev", vp), ("retrieve_dev", vp),
        ("n_paths", C.c_int32), ("depth", C.c_int32), ("n_nodes_dev", vp), ("n_paths_dev", vp), ("done_dev", vp),
        ("slots_dev", vp), ("n_slots", C.c_int32), ("counts_dev", vp), ("repetition_dev", vp), ("presence_dev", vp),
        ("frequency_dev", vp),
    ]


class StopArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("width", C.c_int32), ("tokens_dev", vp), ("count_dev", vp), ("hist_dev", vp),
        ("hist_stride", C.c_int32), ("hist_len_dev", vp), ("stop_tokens_dev", vp), ("stop_len_dev", vp), ("done_dev", vp),
        ("out_count_dev", vp), ("out_hit_dev", vp),
    ]


class LogitControlArgs(C.Structure):
    _fields_ = [
        ("logits_dev", vp), ("dtype", C.c_int32), ("batch", C.c_int32), ("n_nodes", C.c_int32), ("vocab", C.c_int32),
        ("batch_stride", C.c_int64), ("row_stride", C.c_int64), ("tokens_dev", vp), ("retrieve_dev", vp),
        ("n_paths", C.c_int32), ("depth", C.c_int32), ("n_nodes_dev", vp), ("n_paths_dev", vp), ("done_dev", vp),
        ("slots_dev", vp), ("n_slots", C.c_int32), ("hist_dev", vp), ("hist_stride", C.c_int32), ("hist_len_dev", vp),
        ("bias_ids_dev", vp), ("bias_dev", vp), ("bias_n_dev", vp), ("bad_tokens_dev", vp), ("bad_len_dev", vp),
        ("min_tokens_dev", vp), ("stop_tokens_dev", vp), ("stop_len_dev", vp), ("eos_token", C.c_int32),
    ]


class AssembleArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("n_nodes", C.c_int32), ("n_paths", C.c_int32), ("depth", C.c_int32), ("type_dev", vp),
        ("draft_dev", vp), ("draft_stride", C.c_int32), ("draft_len_dev", vp), ("tree_tokens_dev", vp),
        ("tree_parents_dev", vp), ("tree_depth_dev", vp), ("tree_stride", C.c_int32), ("tree_n_dev", vp),
        ("tree_retrieve_dev", vp), ("tree_max_paths", C.c_int32), ("tree_max_depth", C.c_int32), ("tree_shape_dev", vp),
        ("cache_len_dev", vp), ("done_dev", vp), ("mask_dtype", C.c_int32), ("kv_len", C.c_int32),
        ("out_tokens_dev", vp), ("out_position_ids_dev", vp), ("out_n_nodes_dev", vp), ("out_n_paths_dev", vp),
        ("out_retrieve_dev", vp), ("out_mask_dev", vp),
    ]


# name -> (restype, argtypes); every symbol include/samd_b200.h declares
SYMBOLS = {
    "samd_abi_version": (C.c_int, []),
    "samd_last_error": (C.c_char_p, []),
    "samd_device_count": (C.c_int, []),
    "samd_launch_count": (C.c_int64, []),
    "samd_dyn_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(vp)]),
    "samd_dyn_destroy": (C.c_int, [vp]),
    "samd_dyn_reset": (C.c_int, [vp, vp, vp]),
    "samd_dyn_bytes": (C.c_int64, [vp]),
    "samd_dyn_copy": (C.c_int, [vp, vp, vp]),
    "samd_dyn_clone": (C.c_int, [vp, vp, vp, vp, C.c_int32, vp]),
    "samd_dyn_grow": (C.c_int, [vp, C.c_int, C.POINTER(vp)]),
    "samd_dyn_stats": (C.c_int, [vp, c_i64p]),
    "samd_dyn_meta": (C.c_int, [vp, c_i32p]),
    "samd_dyn_export": (C.c_int, [vp, C.c_int, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p, C.c_int64]),
    "samd_dyn_export_edges": (C.c_int, [vp, C.c_int, c_i32p, C.c_int64]),
    "samd_dyn_gen_draft": (C.c_int, [vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_double, vp, C.c_int32, vp, vp]),
    "samd_static_from_arrays": (C.c_int, [C.c_int64, c_i32p, c_i32p, c_i32p, c_i32p, C.c_int64, c_i32p, C.c_int64, c_i32p,
                                          C.POINTER(vp)]),
    "samd_static_export_edges": (C.c_int, [vp, c_i32p, c_i32p]),
    "samd_static_gen_draft": (C.c_int, [vp, vp, vp, C.c_int, C.c_int32, vp, C.c_int32, vp]),
    "samd_static_build": (C.c_int, [c_i32p, c_i64p, C.c_int64, C.c_int32, C.c_int, C.POINTER(vp)]),
    "samd_static_build_host": (C.c_int, [c_i32p, c_i64p, C.c_int64, C.c_int32, C.c_int, C.POINTER(vp)]),
    "samd_static_upload": (C.c_int, [vp]),
    "samd_static_drop_host": (C.c_int, [vp]),
    "samd_static_destroy": (C.c_int, [vp]),
    "samd_static_info": (C.c_int, [vp, c_i64p]),
    "samd_static_export": (C.c_int, [vp, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p]),
    "samd_static_save": (C.c_int, [vp, C.c_char_p]),
    "samd_static_load": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
    "samd_static_load_host": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
    "samd_static_set_l2_window": (C.c_int, [vp, vp, C.c_int64]),
    "samd_step": (C.c_int, [C.POINTER(StepArgs), vp]),
    "samd_step_set_debug_cycles": (None, [vp]),
    "samd_step_set_scouts": (None, [C.c_int]),
    "samd_step_set_variant": (None, [C.c_int]),
    "samd_step_set_prewalk": (None, [C.c_int]),
    "samd_step_set_ngram": (None, [C.c_int]),
    "samd_step_set_lean": (None, [C.c_int]),
    "samd_step_set_trace": (None, [vp, C.c_int]),
    "samd_stage_copy": (C.c_int, [vp, vp, C.c_int64, vp]),
    "samd_debug_granule_copy": (C.c_int, [vp, vp, vp, C.c_int64, C.c_int32, C.c_int32, vp]),
    "samd_debug_warp_slots": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp]),
    "samd_debug_replay_trace": (C.c_int, [vp, vp, C.c_int, C.c_int, vp, vp]),
    "samd_static_tree_draft": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, C.c_int32, C.c_double, C.c_int32, C.c_int32,
                                         vp, vp, vp, vp, vp, C.c_int32, C.c_int32, vp, vp]),
    "samd_draft_assemble": (C.c_int, [C.POINTER(AssembleArgs), vp]),
    "samd_static_lookup_keys": (C.c_int, [vp, vp, vp, C.c_int, C.c_int64, vp, vp]),
    "samd_draft_from_keys": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int, C.c_int32, vp, vp, C.c_int32, vp]),
    "samd_xchg_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "samd_xchg_export": (C.c_int, [vp, vp]),
    "samd_xchg_connect": (C.c_int, [vp, vp]),
    "samd_xchg_destroy": (C.c_int, [vp]),
    "samd_xchg_status": (C.c_int, [vp]),
    "samd_static_lookup_exchange": (C.c_int, [vp, vp, vp, C.c_int32, vp, vp, C.c_int64, vp, vp]),
    "samd_draft_from_exchange": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int32, vp, vp, C.c_int32, vp]),
    "samd_static_walk": (C.c_int, [vp, vp, vp, C.c_int32, vp, vp, C.c_int, vp, vp, vp]),
    "samd_dyn_transfer": (C.c_int, [vp, vp, C.c_int32, vp, vp]),
    "samd_kv_compact": (C.c_int, [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64, vp, C.c_int32,
                                  vp, vp, C.c_int32, vp]),
    "samd_kv_copy_rows": (C.c_int, [vp, C.c_int64, C.c_int64, C.c_int64, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                                    C.c_int32, C.c_int32, vp, vp, vp, C.c_int32, vp]),
    "samd_debug_pointer_chase": (C.c_int, [vp, C.c_int64, C.c_int, C.c_int, vp, vp]),
    "samd_verify_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(vp)]),
    "samd_verify_destroy": (C.c_int, [vp]),
    "samd_verify_compact": (C.c_int, [vp, C.POINTER(VerifyArgs), vp]),
    "samd_verify_sample": (C.c_int, [C.POINTER(SampleArgs), vp]),
    "samd_verify_sample_requests": (C.c_int, [C.POINTER(SampleArgs), C.POINTER(SampleRequestArgs), vp]),
    "samd_token_logprobs": (C.c_int, [C.POINTER(LogprobArgs), vp]),
    "samd_apply_penalties": (C.c_int, [C.POINTER(PenaltyArgs), vp]),
    "samd_stop_match": (C.c_int, [C.POINTER(StopArgs), vp]),
    "samd_apply_logit_controls": (C.c_int, [C.POINTER(LogitControlArgs), vp]),
    "samd_recycle_gen_tree": (C.c_int, [vp, C.c_int32, vp, vp, C.c_int32, vp, vp, C.c_int32, C.c_int32, vp, vp]),
    "samd_verify_set_chunk": (None, [C.c_int]),
    "samd_verify_set_overlap": (None, [C.c_int]),
    "samd_verify_set_even_items": (None, [C.c_int]),
    "samd_verify_set_tma": (None, [C.c_int]),
    "samd_verify_set_debug_times": (None, [C.c_void_p]),
}

_lib = None


class SamdError(RuntimeError):
    pass


def lib():
    """Load libsamd_b200.so once; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SamdError(
                f"{LIB_PATH} not found: build it with `python __graft_entry__.py build` "
                "(the SAM-Decoding hot path has no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
        if _lib.samd_abi_version() != 3:
            raise SamdError("libsamd_b200.so ABI version mismatch")
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().samd_last_error().decode("utf-8", "replace")
        raise SamdError(f"{what or 'samd call'} failed (rc={rc}): {msg}")


def require_device():
    if lib().samd_device_count() <= 0:
        raise SamdError("no CUDA device: the SAM-Decoding hot path runs on the GPU only (no CPU fallback)")


def ptr(t):
    """Device (or host) pointer of a torch tensor / None."""
    return None if t is None else t.data_ptr()


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream
