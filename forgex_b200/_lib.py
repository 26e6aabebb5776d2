"""ctypes binding of libforgex_b200.so (the C ABI of include/forgex_b200.h).

The library must have been built in-tree (python -m forgex_b200.build or __graft_entry__.build()).
Loading fails loudly when it is missing: there is no Python or CPU fallback for the matching path.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libforgex_b200.so")

FX_OP_MATCH, FX_OP_IN, FX_OP_REGEX = 0, 1, 2
FX_TABLE_AUTO, FX_TABLE_SMEM, FX_TABLE_GLOBAL = 0, 1, 2
FX_ERR_TREE_NODE_LIMIT, FX_ERR_DFA_STATE_CAP, FX_ERR_PREFILTER_UNSUPPORTED = 101, 102, 103
FX_ERR_BAD_ARGUMENT, FX_ERR_NO_DEVICE, FX_ERR_WORK_BUDGET = 104, 105, 106
FX_STATEMAP_MAP_WORDS, FX_STATEMAP_UNKNOWN = 98, -2
FX_STATEMAP_WALK_WORDS, FX_STATEMAP_WALK_NEW, FX_STATEMAP_WALK_DONE = 4, -1, -2

# every symbol include/forgex_b200.h declares (tests check that the library exports them all)
SYMBOLS = [
    "fx_status_message", "fx_compile", "fx_compile_from_dfa", "fx_pattern_cp_automaton", "fx_pattern_free", "fx_pattern_get_info", "fx_pattern_set_residency",
    "fx_pattern_literals", "fx_pattern_tables", "fx_pattern_span_tables", "fx_pattern_nfa_tables", "fx_is_valid_regex", "fx_is_valid_regex_batch",
    "fx_match_fixed_dev", "fx_in_fixed_dev", "fx_match_batch_dev", "fx_in_batch_dev", "fx_regex_batch_dev",
    "fx_regex_buffer_work_bytes", "fx_regex_buffer_dev", "fx_buffer_scan_dev", "fx_buffer_scan_all_dev", "fx_buffer_finish_dev",
    "fx_statemap_window_dev", "fx_statemap_combine", "fx_statemap_back_dev",
    "fx_match_fixed", "fx_in_fixed", "fx_match_batch", "fx_in_batch", "fx_regex_batch", "fx_regex_buffer",
    "fx_regex_count_batch_dev", "fx_regex_buffer_all_dev", "fx_regex_count_batch", "fx_regex_buffer_all",
    "fx_in", "fx_match", "fx_regex", "fx_in_value", "fx_match_value", "fx_regex_sub", "fx_launch_count",
]


class PatternInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "op", "status", "nfa_states", "cp_states", "cp_classes", "byte_states", "byte_classes", "row_shift",
        "table_bytes", "direct_bytes", "literal_all_len", "literal_prefix_len", "literal_suffix_len",
        "literal_only", "residency", "direct", "prefix_mode", "sparse", "sparse_ranges")] + [
        ("sparse_lo", C.c_int32 * 4), ("sparse_hi", C.c_int32 * 4), ("sparse_high", C.c_int32),
        ("sparse_second", C.c_int32), ("sparse_used", C.c_int32), ("prefix_scan", C.c_int32), ("statemap", C.c_int32),
        ("nfa_engine", C.c_int32), ("compact_used", C.c_int32), ("statemap_used", C.c_int32), ("gated", C.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO):
        raise ImportError("forgex_b200: %s is missing -- build it with `python -m forgex_b200.build` "
                          "(there is no CPU fallback for the matching path)" % SO)
    L = C.CDLL(SO)
    vp, i64, u8p = C.c_void_p, C.c_int64, C.c_void_p
    L.fx_status_message.restype = C.c_char_p
    L.fx_status_message.argtypes = [C.c_int]
    L.fx_compile.argtypes = [C.c_char_p, i64, C.c_int, C.POINTER(vp)]
    L.fx_pattern_free.argtypes = [vp]
    L.fx_compile_from_dfa.argtypes = [C.c_int, vp, C.c_int32, vp, C.c_int32, vp, C.c_int32, C.c_char_p, i64, C.c_char_p, i64,
                                      C.c_char_p, i64, C.POINTER(vp)]
    L.fx_pattern_cp_automaton.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int32 * 4)]
    L.fx_in_value.argtypes = [C.c_char_p, i64, C.c_char_p, i64]
    L.fx_match_value.argtypes = [C.c_char_p, i64, C.c_char_p, i64]
    L.fx_regex_sub.restype = None
    L.fx_regex_sub.argtypes = [C.c_char_p, i64, C.c_char_p, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64),
                               C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.fx_pattern_get_info.argtypes = [vp, C.POINTER(PatternInfo)]
    L.fx_pattern_set_residency.argtypes = [vp, C.c_int]
    L.fx_pattern_literals.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_char_p]
    L.fx_pattern_tables.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp),
                                    C.POINTER(C.c_int32 * 6)]
    L.fx_pattern_span_tables.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int32 * 4), C.POINTER(vp),
                                         C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int32 * 4)]
    L.fx_pattern_nfa_tables.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int32 * 5)]
    L.fx_is_valid_regex.argtypes = [C.c_char_p, i64, C.POINTER(C.c_int)]
    L.fx_is_valid_regex_batch.argtypes = [vp, vp, i64, vp, vp]
    for name in ("fx_match_fixed_dev", "fx_in_fixed_dev"):
        getattr(L, name).argtypes = [vp, u8p, i64, i64, u8p, vp]
    for name in ("fx_match_batch_dev", "fx_in_batch_dev"):
        getattr(L, name).argtypes = [vp, u8p, vp, i64, i64, u8p, vp]
    L.fx_regex_batch_dev.argtypes = [vp, u8p, vp, i64, i64, vp, vp, vp]
    L.fx_regex_buffer_work_bytes.restype = i64
    L.fx_regex_buffer_work_bytes.argtypes = [i64]
    L.fx_regex_buffer_dev.argtypes = [vp, u8p, i64, vp, vp, vp]
    L.fx_buffer_scan_dev.argtypes = [vp, u8p, i64, i64, i64, i64, C.c_int, C.c_int, vp, vp]
    L.fx_buffer_scan_all_dev.argtypes = [vp, u8p, i64, i64, i64, i64, C.c_int, C.c_int, vp, vp]
    L.fx_buffer_finish_dev.argtypes = [vp, u8p, i64, i64, C.c_int, vp, vp, vp]
    L.fx_statemap_window_dev.argtypes = [vp, u8p, i64, i64, i64, i64, vp, vp, vp]
    L.fx_statemap_combine.argtypes = [vp, vp, i64, i64, vp]
    L.fx_statemap_back_dev.argtypes = [vp, u8p, i64, i64, i64, vp, vp]
    for name in ("fx_match_fixed", "fx_in_fixed"):
        getattr(L, name).argtypes = [vp, u8p, i64, i64, u8p]
    for name in ("fx_match_batch", "fx_in_batch"):
        getattr(L, name).argtypes = [vp, u8p, vp, i64, u8p]
    L.fx_regex_batch.argtypes = [vp, u8p, vp, i64, vp, vp]
    L.fx_regex_buffer.argtypes = [vp, u8p, i64, C.POINTER(i64), C.POINTER(i64)]
    L.fx_regex_count_batch_dev.argtypes = [vp, u8p, vp, i64, i64, vp, vp]
    L.fx_regex_buffer_all_dev.argtypes = [vp, u8p, i64, vp, vp, i64, C.POINTER(i64), vp, vp]
    L.fx_regex_count_batch.argtypes = [vp, u8p, vp, i64, vp]
    L.fx_regex_buffer_all.argtypes = [vp, u8p, i64, vp, vp, i64, C.POINTER(i64)]
    L.fx_in.argtypes = [C.c_char_p, i64, C.c_char_p, i64, C.POINTER(C.c_int)]
    L.fx_match.argtypes = [C.c_char_p, i64, C.c_char_p, i64, C.POINTER(C.c_int)]
    L.fx_regex.argtypes = [C.c_char_p, i64, C.c_char_p, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64),
                           C.POINTER(C.c_int)]
    L.fx_launch_count.restype = i64
    L.fx_launch_count.argtypes = []
    _lib = L
    return L
