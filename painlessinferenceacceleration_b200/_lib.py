# -*- coding: utf-8 -*-
"""ctypes binding of libpia_b200.so (include/pia_b200.h). The product path has no CPU fallback: a missing
library or a missing CUDA device raises."""
import ctypes as C
import os

from .build import SO

_lib = None

i32p = C.POINTER(C.c_int32)
u64p = C.POINTER(C.c_uint64)
vp = C.c_void_p

PIA_OK, PIA_ERR_INVALID, PIA_ERR_INDEX, PIA_ERR_CAPACITY, PIA_ERR_CUDA, PIA_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
MODE = {'input': 0, 'output': 1, 'mix': 2}
GET_HIER, GET_ONE = 0, 1
GET_TAIL = 1
GET_FIRST_ONLY = 2


class TrieConfig(C.Structure):
    _fields_ = [('vocab_capacity', C.c_int32), ('node_capacity', C.c_int64), ('edge_capacity', C.c_int64),
                ('n_input_slots', C.c_int32), ('max_node', C.c_int32), ('max_output_node', C.c_int32),
                ('max_put_tokens', C.c_int32), ('frontier_capacity', C.c_int32), ('max_resident_queries', C.c_int32)]


class TrieStats(C.Structure):
    _fields_ = [('nodes_used', C.c_int64), ('edges_used', C.c_int64), ('n_trees', C.c_int32),
                ('n_update_trees', C.c_int32), ('n_update_input_trees', C.c_int32), ('error_flags', C.c_int32),
                ('nodes_visited', C.c_int64), ('edges_visited', C.c_int64)]


class AttnConfig(C.Structure):
    _fields_ = [('n_q_heads', C.c_int32), ('n_kv_heads', C.c_int32), ('head_dim', C.c_int32), ('max_seq', C.c_int32),
                ('max_nodes', C.c_int32), ('n_layers', C.c_int32), ('kv_split_max', C.c_int32), ('n_slots', C.c_int32)]


class AcceptConfig(C.Structure):
    _fields_ = [('vocab', C.c_int32), ('max_nodes', C.c_int32), ('repetition_penalty', C.c_float),
                ('n_eos', C.c_int32), ('eos', C.c_int32 * 8), ('max_length', C.c_int32), ('bound_walk', C.c_int32)]


class Slots(C.Structure):
    """pia_slots_t: the request slots of one verify step (device arrays, read at kernel run time)"""
    _fields_ = [('batch', C.c_int32), ('rows_per_slot', C.c_int32), ('d_n', C.c_void_p), ('d_prefix_len', C.c_void_p),
                ('d_pad_len', C.c_void_p), ('kv_slot_stride', C.c_int64), ('kv_first_slot', C.c_int32)]


# every symbol include/pia_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    'pia_last_error': (C.c_char_p, []),
    'pia_abi_version': (C.c_int, []),
    'pia_launch_count': (C.c_ulonglong, []),
    'pia_trie_create': (C.c_int, [C.POINTER(TrieConfig), C.POINTER(vp)]),
    'pia_trie_destroy': (C.c_int, [vp]),
    'pia_trie_set_eos': (C.c_int, [vp, i32p, C.c_int]),
    'pia_trie_set_stop_words': (C.c_int, [vp, i32p, C.c_int]),
    'pia_trie_set_limits': (C.c_int, [vp, C.c_int, C.c_int]),
    'pia_trie_put': (C.c_int, [vp, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    'pia_trie_tree_put': (C.c_int, [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp]),
    'pia_trie_stream_put': (C.c_int, [vp, vp, C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, vp]),
    'pia_trie_get': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]),
    'pia_trie_tree_squeeze': (C.c_int, [vp, C.c_int, vp]),
    'pia_trie_tree_reset_input_freq': (C.c_int, [vp, C.c_int, C.c_int, vp]),
    'pia_trie_reset_input_freqs': (C.c_int, [vp, C.c_int, vp]),
    'pia_trie_squeeze_branch_counts': (C.c_int, [vp, vp]),
    'pia_trie_fresh': (C.c_int, [vp, vp]),
    'pia_trie_stats': (C.c_int, [vp, C.POINTER(TrieStats), vp]),
    'pia_trie_copy_error_flags': (C.c_int, [vp, vp, vp]),
    'pia_trie_tree_counters': (C.c_int, [vp, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), vp]),
    'pia_trie_compact': (C.c_int, [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), vp]),
    'pia_trie_export_sizes': (C.c_int, [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), vp]),
    'pia_trie_export': (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, vp, vp, vp, vp]),
    'pia_trie_import': (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, vp, vp, vp, vp]),
    'pia_attn_plan_create': (C.c_int, [C.POINTER(AttnConfig), vp, vp, C.POINTER(vp)]),
    'pia_attn_plan_destroy': (C.c_int, [vp]),
    'pia_attn_plan_set_debug': (C.c_int, [vp, vp]),
    'pia_attn_plan_grid': (C.c_int, [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'pia_tree_attn_fwd': (C.c_int, [vp, C.c_int, vp, vp, C.POINTER(Slots), C.c_float, vp, vp]),
    'pia_tree_attn_fused_fwd': (C.c_int, [vp, C.c_int, vp, vp, vp, C.c_int, vp, C.POINTER(Slots), C.c_float, vp, vp]),
    'pia_rmsnorm': (C.c_int, [vp, vp, vp, C.c_float, C.c_int, C.c_int, vp, vp, vp]),
    'pia_rmsnorm_partials': (C.c_int, [vp, C.c_int, C.c_int64, vp, vp, C.c_float, C.c_int, C.c_int, vp, vp, vp]),
    'pia_gemm_plan_create': (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    'pia_gemm_plan_create_grouped': (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.POINTER(vp)]),
    'pia_gemm_plan_create_fp8': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.POINTER(vp)]),
    'pia_gemm_plan_create_grouped_fp8': (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.POINTER(vp)]),
    'pia_gemm_plan_destroy': (C.c_int, [vp]),
    'pia_gemm_plan_splits': (C.c_int, [vp]),
    'pia_gemm_plan_set_pdl': (C.c_int, [vp, C.c_int]),
    'pia_gemm_plan_set_silu': (C.c_int, [vp, C.c_int]),
    'pia_gemm_run': (C.c_int, [vp, C.c_int, vp, vp]),
    'pia_rope_kv_append': (C.c_int, [vp, vp, C.c_int, C.POINTER(Slots), C.c_int, C.c_int, C.c_int, vp, vp,
                                     C.c_int, vp, vp, vp, C.c_int, vp]),
    'pia_silu_mul': (C.c_int, [vp, C.c_int, C.c_int, vp, vp]),
    'pia_embed_gather': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, vp, vp]),
    'pia_moe_combine': (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    'pia_moe_router': (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    'pia_l2_prefetch': (C.c_int, [vp, C.c_int64, C.c_int64, C.c_int64, C.c_float, vp]),
    'pia_accept': (C.c_int, [C.POINTER(AcceptConfig), vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int, vp,
                             vp, vp, vp, vp, vp, vp, vp, vp]),
    'pia_accept_workspace_bytes': (C.c_int64, [C.POINTER(AcceptConfig)]),
    'pia_kv_compact': (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, vp, C.c_int, vp, vp,
                                 vp]),
    'pia_flood_update_draft_table': (C.c_int, [vp, C.c_int, vp, vp, C.c_int64, C.c_int, C.c_int, C.c_int, vp]),
    'pia_flood_retrieve_draft_table': (C.c_int, [vp, C.c_int, vp, vp, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, vp,
                                                 vp]),
    'pia_flood_verify_draft': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    'pia_flood_update_draft_cache': (C.c_int, [vp, C.c_int64, vp, vp, C.c_int, vp]),
}


def load():
    """dlopen libpia_b200.so and type every entry point. Raises if the library is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            raise RuntimeError(f'{SO} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                               '(there is no CPU fallback)')
        L = C.CDLL(SO)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class PiaError(RuntimeError):
    pass


def check(rc):
    if rc == PIA_OK:
        return
    msg = load().pia_last_error().decode(errors='replace')
    if rc == PIA_ERR_INVALID:
        raise AssertionError(msg)
    if rc == PIA_ERR_INDEX:
        raise IndexError('list index out of range')
    raise PiaError(f'libpia_b200 error {rc}: {msg}')
