"""ctypes binding of the C-ABI library declared in ``include/genlm_trie_b200.h``.

There is no Python or CPU fallback behind these calls: if the shared library is missing and cannot be
compiled, importing this module raises.
"""
import ctypes
import os

from . import build as _build

c_void_p, c_int, c_int32, c_int64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64
c_uint, c_uint64, c_size_t, c_float, c_char_p = ctypes.c_uint, ctypes.c_uint64, ctypes.c_size_t, ctypes.c_float, ctypes.c_char_p

GT_F32, GT_F64, GT_F16, GT_BF16 = 0, 1, 2, 3
GT_OP_SUM, GT_OP_MAX = 1, 2
GT_FLAG_LOG_INPUT = 1
GT_FLAG_DFS_ORDER = 2
GT_FLAG_PHASE_PERMUTE, GT_FLAG_PHASE_TILE, GT_FLAG_PHASE_SPAN = 0x100, 0x200, 0x400
GT_GATHER_LOG = 1
GT_CHILD_NORMALIZE, GT_CHILD_LOG = 0x10, 0x20
GT_MASK_NONE, GT_MASK_ADD_F32, GT_MASK_BOOL_U8, GT_MASK_BITS_U32 = 0, 1, 2, 3
GT_RESAMPLE_MULTINOMIAL, GT_RESAMPLE_STRATIFIED, GT_RESAMPLE_SYSTEMATIC = 0, 1, 2
GT_RESAMPLE_MAX_GROUP = 16384
GT_PDA_POP, GT_PDA_MAX_DEPTH = -2, 64


class PlanInfo(ctypes.Structure):
    _fields_ = [
        ("n_tokens", c_int64), ("n_nodes", c_int64),
        ("tile_leaves", c_int32), ("n_tiles", c_int32), ("rows_per_item", c_int32), ("permute_unit", c_int32),
        ("n_span", c_int32), ("max_levels", c_int32), ("span_terms", c_int64),
        ("max_tile_values", c_int32), ("reserved", c_int32),
        ("staged_slots", c_int64), ("meta_bytes", c_int64),
    ]


# name -> (restype, argtypes); every symbol include/genlm_trie_b200.h declares
SIGNATURES = {
    "gt_last_error": (c_char_p, []),
    "gt_version": (c_int, []),
    "gt_build": (c_int, [c_void_p, c_void_p, c_int64, ctypes.POINTER(c_void_p)]),
    "gt_free": (None, [c_void_p]),
    "gt_num_tokens": (c_int64, [c_void_p]),
    "gt_num_nodes": (c_int64, [c_void_p]),
    "gt_root": (c_int64, [c_void_p]),
    "gt_num_reach": (c_int64, [c_void_p]),
    "gt_max_depth": (c_int64, [c_void_p]),
    "gt_export_layout": (c_int, [c_void_p] * 9),
    "gt_export_reachability": (c_int, [c_void_p, c_void_p, c_void_p]),
    "gt_upload": (c_int, [c_void_p, c_int]),
    "gt_get_plan_info": (c_int, [c_void_p, ctypes.POINTER(PlanInfo)]),
    "gt_plan": (c_int, [c_void_p, c_int32]),
    "gt_export_plan_array": (c_int64, [c_void_p, c_char_p, c_void_p, c_int64, ctypes.POINTER(c_int32)]),
    "gt_debug_read_trace": (c_int64, [c_void_p, c_int, c_void_p, c_int64, c_void_p]),
    "gt_workspace_bytes": (c_size_t, [c_void_p, c_int64]),
    "gt_weight_reduce": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int, c_int64,
                                 c_uint, c_uint, c_void_p, c_size_t, c_void_p]),
    "gt_gather_nodes": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_uint,
                                c_void_p, c_int64, c_void_p]),
    "gt_download_rows": (c_int, [c_void_p, c_size_t, c_void_p, c_size_t, c_size_t, c_int64, c_void_p]),
    "gt_subtree_token_mask": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "gt_max_children": (c_int64, [c_void_p]),
    "gt_child_workspace_bytes": (c_size_t, [c_void_p, c_int64]),
    "gt_child_masses": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                c_uint, c_uint, c_void_p, c_size_t, c_void_p]),
    "gt_child_sample": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_uint, c_uint64, c_uint64, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gt_num_symbols": (c_int64, [c_void_p]),
    "gt_symbol_masses": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                                 c_uint, c_uint, c_void_p, c_size_t, c_void_p]),
    "gt_symbol_sample": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_uint, c_uint64,
                                 c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gt_child_masses_masked": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                       c_void_p, c_void_p, c_int64, c_uint, c_uint, c_void_p, c_size_t, c_void_p]),
    "gt_child_sample_masked": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_uint,
                                       c_uint64, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gt_symbol_masses_masked": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                        c_void_p, c_int64, c_uint, c_uint, c_void_p, c_size_t, c_void_p]),
    "gt_symbol_sample_masked": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                        c_int64, c_uint, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_size_t, c_void_p]),
    "gt_dfa_token_mask": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                  c_void_p]),
    "gt_dfa_token_logw": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                  c_int64, c_void_p]),
    "gt_dfa_advance": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                               c_void_p]),
    "gt_pda_token_mask": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                  c_int64, c_void_p, c_int64, c_void_p]),
    "gt_pda_token_logw": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64,
                                  c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "gt_pda_advance": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                               c_void_p, c_int64, c_void_p, c_void_p]),
    "gt_lse_sample": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_int, c_int64, c_float,
                              c_uint64, c_uint64, c_void_p, c_void_p, c_void_p]),
    "gt_resample": (c_int, [c_void_p, c_int64, c_int64, c_int, c_float, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p,
                            c_void_p, c_void_p, c_void_p]),
}


def _load():
    path = _build.LIB_PATH
    if not os.path.exists(path) or (os.environ.get("GT_AUTO_REBUILD") == "1" and _build.needs_build()):
        # building is part of installing the package, not a fallback: it produces the CUDA library
        _build.build()
    lib = ctypes.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


lib = _load()


class GtError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        msg = lib.gt_last_error()
        raise GtError(f"{what} failed (status {rc}): {msg.decode() if msg else '?'}")
