"""The C-ABI library loads and exports every symbol include/sxcross.h declares (no GPU needed)."""
import ctypes
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "sxcross.h")
LIB = os.path.join(ROOT, "smart-crossover_b200", "libsxcross.so")


def _declared():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"SX_API[^;(]*?\b(sx_[a-z0-9_]+)\s*\(", src)))


def _ensure_built():
    if not os.path.exists(LIB):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "smart-crossover_b200", "csrc"), "-j8"])


def test_header_declares_the_expected_entry_points():
    names = _declared()
    for must in ("sx_score_ot", "sx_score_mcf", "sx_argsort_f64", "sx_kruskal_order", "sx_kruskal",
                 "sx_tree_potentials", "sx_price_pass_begin", "sx_price_dense_ot", "sx_price_arcs", "sx_topk_select",
                 "sx_exchange_blocks", "sx_topk_merge", "sx_price_dense_ot_h"):
        assert must in names
    assert len(names) >= 24


def test_library_exports_every_declared_symbol_at_abi_6():
    _ensure_built()
    lib = ctypes.CDLL(LIB)
    for name in _declared():
        assert hasattr(lib, name), f"{name} declared in sxcross.h but not exported"
    lib.sx_abi_version.restype = ctypes.c_int
    assert lib.sx_abi_version() == 6
    lib.sx_error_string.restype = ctypes.c_char_p
    assert b"spanning" in lib.sx_error_string(-5)


def test_binding_signatures_cover_the_header():
    _ensure_built()
    import smart_crossover._native as native
    assert sorted(native.SIGNATURES) == _declared()


def test_workspace_queries_and_argument_validation_without_gpu():
    """Pure host-side entry points: sizes are monotone, bad arguments are rejected before any CUDA call."""
    _ensure_built()
    import smart_crossover._native as native
    lib = native.lib
    assert lib.sx_argsort_workspace_bytes(1000) < lib.sx_argsort_workspace_bytes(10**6)
    assert lib.sx_kruskal_workspace_bytes(80, 1600) > 0
    assert lib.sx_tree_potentials_workspace_bytes(80) > 0
    assert lib.sx_topk_workspace_bytes(1 << 20, 1024) > 0
    assert lib.sx_score_ot(None, None, None, 3, 3, None, None, None) == -1
    assert lib.sx_argsort_f64(None, 10, None, None, None, 0, None) == -1
    assert lib.sx_price_dense_ot(None, 4, 0, 4, 4, None, None, 1e-6, None, None, None, None, 0, None, 0, -1, None) == -1
    assert lib.sx_select_state_bytes() >= 2 * 1024 * 1024
    assert lib.sx_price_pass_begin(None, None, 16, None) == -1
    assert lib.sx_key_to_f64(0x7fffffffffffffff) != lib.sx_key_to_f64(0x7fffffffffffffff)  # NaN image of the reset value
