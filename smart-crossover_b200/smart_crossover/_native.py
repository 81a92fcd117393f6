"""ctypes binding of libsxcross.so (the C ABI declared in include/sxcross.h).

There is no CPU fallback: if the library is missing the import raises, and every
call checks the returned status and raises `SxError`.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libsxcross.so")

SX_OK = 0
SX_ERR_NOT_SPANNING = -5
SX_ERR_UNALIGNED = -6
SX_ERR_WORKSPACE = -3
SX_ERR_PUSH_ASSERT = -9
SX_PLUS_IS_HEAD = 0
SX_PLUS_IS_TAIL = 1
SX_TOPK_MAX_K = 1024
SX_STATUS_CAND_OVERFLOW = 1
SX_STATUS_DUPLICATE_CANDIDATES = 2
SX_STATUS_K_MISMATCH = 4
SX_STATUS_NAN_RC = 8
SX_STATUS_REPEAT_MASK = 1
SX_ABI_VERSION = 6


class SxError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        detail = lib.sx_error_string(code).decode()
        if code == -2:
            detail += f" [cudaError {lib.sx_last_cuda_error()}]"
        super().__init__(f"{where}: {detail} ({code})")


class PriceHeader(ctypes.Structure):
    _fields_ = [("n_violating", ctypes.c_ulonglong), ("min_rc_key", ctypes.c_longlong),
                ("n_priced", ctypes.c_ulonglong), ("status", ctypes.c_ulonglong)]


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C smart-crossover_b200/csrc`. There is no CPU fallback for the device path.")

lib = ctypes.CDLL(LIB_PATH)

_p = ctypes.c_void_p
_i64 = ctypes.c_int64
_sz = ctypes.c_size_t
_int = ctypes.c_int
_dbl = ctypes.c_double

# name -> (restype, argtypes); mirrors include/sxcross.h one to one
SIGNATURES = {
    "sx_abi_version": (_int, []),
    "sx_error_string": (ctypes.c_char_p, [_int]),
    "sx_last_cuda_error": (_int, []),
    "sx_key_to_f64": (_dbl, [ctypes.c_longlong]),
    "sx_score_ot": (_int, [_p, _p, _p, _i64, _i64, _p, _p, _p]),
    "sx_score_mcf_workspace_bytes": (_sz, [_i64, _i64]),
    "sx_score_mcf": (_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _i64, _p, _p, _sz, _p]),
    "sx_sort_set_tuning": (_int, [_int]),
    "sx_score_set_tuning": (_int, [_int]),
    "sx_kruskal_set_tuning": (_int, [_int]),
    "sx_argsort_workspace_bytes": (_sz, [_i64]),
    "sx_argsort_f64": (_int, [_p, _i64, _p, _p, _p, _sz, _p]),
    "sx_argsort_u64": (_int, [_p, _i64, _int, _p, _p, _p, _sz, _p]),
    "sx_queue_from_order": (_int, [_p, _i64, _p, _p]),
    "sx_kruskal_order_workspace_bytes": (_sz, [_i64]),
    "sx_kruskal_order": (_int, [_p, _p, _i64, _p, _p, _sz, _p]),
    "sx_kruskal_order_head": (_int, [_p, _p, _i64, _i64, _i64, _p, _p, _p, _sz, _p]),
    "sx_kruskal_prefix_workspace_bytes": (_sz, [_i64]),
    "sx_hist12_f64": (_int, [_p, _i64, _p, _p]),
    "sx_kruskal_prefix": (_int, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _sz, _p]),
    "sx_kruskal_workspace_bytes": (_sz, [_i64, _i64]),
    "sx_kruskal": (_int, [_p, _i64, _p, _p, _i64, _i64, _i64, _p, _p, _p, _sz, _p]),
    "sx_tree_potentials_workspace_bytes": (_sz, [_i64]),
    "sx_tree_potentials": (_int, [_p, _i64, _p, _p, _i64, _i64, _i64, _p, _i64, _int, _i64, _p, _p, _p, _sz, _p]),
    "sx_select_state_bytes": (_sz, []),
    "sx_tree_flows": (_int, [_p, _i64, _p, _p, _i64, _i64, _i64, _p, _int, _i64, _p, _p, _p, _sz, _p]),
    "sx_price_pass_begin": (_int, [_p, _p, _i64, _p]),
    "sx_price_dense_ot": (_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _dbl, _p, _p, _p, _p, _i64, _p, _i64, _int, _p]),
    "sx_price_arcs": (_int, [_p, _p, _p, _p, _p, _i64, _i64, _dbl, _p, _p, _p, _p, _i64, _p, _p]),
    "sx_price_set_tuning": (_int, [_int, _int]),
    "sx_price_set_tma_options": (_int, [_int, _int]),
    "sx_fused_state_bytes": (_sz, []),
    "sx_fused_state_timestamps_offset": (_sz, []),
    "sx_fused_state_init": (_int, [_p, _i64, _p]),
    "sx_fused_merge_fits": (_int, [_i64, _int]),
    "sx_price_dense_ot_fused": (_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _dbl, _p, _p, _p, _i64, _i64, _p, _i64,
                                       _p, _int, _int, _p, _p, _p, _sz, _p]),
    "sx_topk_workspace_bytes": (_sz, [_i64, _i64]),
    "sx_topk_select": (_int, [_p, _p, _i64, _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "sx_topk_merge_workspace_bytes": (_sz, [_i64]),
    "sx_topk_merge": (_int, [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _p, _i64, _p, _sz, _p]),
    "sx_exchange_buffer_bytes": (_sz, [_i64, _int]),
    "sx_exchange_epoch_offset": (_sz, [_i64, _int]),
    "sx_exchange_blocks": (_int, [_p, _i64, _p, _int, _int, _p, _p]),
    "sx_exchange_ll_buffer_bytes": (_sz, [_i64, _int]),
    "sx_exchange_push_ll": (_int, [_p, _i64, _p, _int, _int, _p]),
    "sx_topk_merge_ll": (_int, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _p]),
    "sx_sinkhorn_workspace_bytes": (_sz, [_i64, _i64]),
    "sx_sinkhorn_ot": (_int, [_p, _i64, _i64, _i64, _p, _p, _dbl, _i64, _dbl, _i64, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "sx_price_dense_ot_h": (_int, [_p, _p, _i64, _i64, _p, _dbl, _i64, _p, _p, _p, _p, _p]),
    "sx_ot_pricer_create": (_int, [_int, _p, _p, _p, _i64, _i64, _i64, _i64, _dbl, _p]),
    "sx_ot_pricer_destroy": (_int, [_p]),
    "sx_ot_pricer_info": (_int, [_p, _int, _p, _p, _p]),
    "sx_ot_pricer_price_h": (_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "sx_ot_pricer_stats": (_int, [_p, _p, _p, _p, _p]),
    "sx_push_tree_h": (_int, [_p, _p, _i64, _i64, _i64, _p, _i64, _p, _p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)   # AttributeError here = header and library out of sync
    _fn.restype = _res
    _fn.argtypes = _args

if lib.sx_abi_version() != SX_ABI_VERSION:
    raise ImportError(f"libsxcross ABI {lib.sx_abi_version()} != binding {SX_ABI_VERSION}")


def check(code, where):
    if code != SX_OK:
        raise SxError(code, where)
