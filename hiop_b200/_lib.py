"""ctypes binding of hiop_b200/libhiopb200.so (declared in include/hiopb200.h).

The library is the product; this file only declares argument types. Loading fails loudly when the shared object is
missing -- there is no Python/CPU fallback for any entry point."""
from __future__ import annotations

import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("HIOPB200_SO") or os.path.join(_HERE, "libhiopb200.so")   # HIOPB200_SO: A/B runs of tools/ against another build
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "hiopb200.h")

HB_OK = 0
HB_FACT_BUNCH_KAUFMAN, HB_FACT_NOPIV, HB_FACT_CHOLESKY = 0, 1, 2

c_dp = ctypes.c_void_p   # device or host pointer to doubles (passed as integer address)
c_ll = ctypes.c_longlong
c_i = ctypes.c_int
c_d = ctypes.c_double
c_vp = ctypes.c_void_p

_lib = None


class EngineError(RuntimeError):
    pass


def declared_symbols() -> list[str]:
    """Every function name declared in include/hiopb200.h (used by the symbol-export test)."""
    txt = open(HEADER_PATH).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(hb_[a-z0-9_]+)\s*\(", txt)))


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise EngineError(f"{SO_PATH} is missing: build it with `make -C hiop_b200/csrc` (or __graft_entry__.build()); "
                          "hiop_b200 has no CPU fallback")
    L = ctypes.CDLL(SO_PATH)
    P = ctypes.POINTER

    def f(name, res, *args):
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = list(args)

    f("hb_version", ctypes.c_char_p)
    f("hb_last_error", ctypes.c_char_p)
    f("hb_launch_count", c_ll)
    f("hb_ctx_create", c_i, c_i, P(c_vp))
    f("hb_ctx_destroy", c_i, c_vp)
    f("hb_ctx_sync", c_i, c_vp)
    f("hb_ctx_phase_timeline", c_i, c_vp, c_i, P(ctypes.c_float))
    f("hb_ctx_stream", c_vp, c_vp)
    f("hb_ctx_device", c_i, c_vp)
    f("hb_ctx_enable_timing", c_i, c_vp, c_i)
    f("hb_ctx_last_syrk_ms", c_i, c_vp, P(ctypes.c_float))
    f("hb_ctx_set_oz_workspace_limit", c_i, c_vp, ctypes.c_size_t)
    f("hb_malloc", c_i, c_vp, ctypes.c_size_t, P(c_vp))
    f("hb_free", c_i, c_vp, c_vp)
    f("hb_malloc_host", c_i, c_vp, ctypes.c_size_t, P(c_vp))
    f("hb_free_host", c_i, c_vp, c_vp)
    f("hb_memcpy_h2d", c_i, c_vp, c_vp, c_vp, ctypes.c_size_t)
    f("hb_memcpy_d2h", c_i, c_vp, c_vp, c_vp, ctypes.c_size_t)
    f("hb_memcpy_d2d", c_i, c_vp, c_vp, c_vp, ctypes.c_size_t)
    f("hb_memset", c_i, c_vp, c_vp, c_i, ctypes.c_size_t)
    f("hb_comm_unique_id", c_i, c_vp)
    f("hb_comm_init", c_i, c_vp, c_i, c_i, c_vp)
    f("hb_comm_size", c_i, c_vp)
    f("hb_comm_rank", c_i, c_vp)
    f("hb_allreduce_sum", c_i, c_vp, c_dp, c_ll)
    # vector ops
    f("hb_vec_set", c_i, c_vp, c_ll, c_dp, c_d)
    f("hb_vec_copy", c_i, c_vp, c_ll, c_dp, c_dp)
    f("hb_vec_scale", c_i, c_vp, c_ll, c_dp, c_d)
    f("hb_vec_axpy", c_i, c_vp, c_ll, c_dp, c_d, c_dp)
    f("hb_vec_axzpy", c_i, c_vp, c_ll, c_dp, c_d, c_dp, c_dp)
    f("hb_vec_axdzpy", c_i, c_vp, c_ll, c_dp, c_d, c_dp, c_dp)
    f("hb_vec_axdzpy_w_pattern", c_i, c_vp, c_ll, c_dp, c_d, c_dp, c_dp, c_dp)
    f("hb_vec_component_mult", c_i, c_vp, c_ll, c_dp, c_dp)
    f("hb_vec_component_div", c_i, c_vp, c_ll, c_dp, c_dp)
    f("hb_vec_component_div_w_pattern", c_i, c_vp, c_ll, c_dp, c_dp, c_dp)
    f("hb_vec_invert", c_i, c_vp, c_ll, c_dp)
    f("hb_vec_select_pattern", c_i, c_vp, c_ll, c_dp, c_dp)
    f("hb_vec_add_constant", c_i, c_vp, c_ll, c_dp, c_d)
    f("hb_vec_add_constant_w_pattern", c_i, c_vp, c_ll, c_dp, c_d, c_dp)
    f("hb_vec_add_log_barrier_grad", c_i, c_vp, c_ll, c_dp, c_d, c_dp, c_dp)
    f("hb_vec_add_linear_damping_term", c_i, c_vp, c_ll, c_dp, c_dp, c_dp, c_d, c_d)
    f("hb_vec_dot", c_i, c_vp, c_ll, c_dp, c_dp, P(c_d))
    f("hb_vec_twonorm", c_i, c_vp, c_ll, c_dp, P(c_d))
    f("hb_vec_infnorm", c_i, c_vp, c_ll, c_dp, P(c_d))
    f("hb_vec_onenorm", c_i, c_vp, c_ll, c_dp, P(c_d))
    f("hb_vec_min_w_pattern", c_i, c_vp, c_ll, c_dp, c_dp, P(c_d))
    f("hb_vec_log_barrier", c_i, c_vp, c_ll, c_dp, c_dp, P(c_d))
    f("hb_vec_linear_damping_term", c_i, c_vp, c_ll, c_dp, c_dp, c_dp, c_d, c_d, P(c_d))
    f("hb_vec_fraction_to_bdry", c_i, c_vp, c_ll, c_dp, c_dp, c_d, c_dp, P(c_d))
    f("hb_mat_times_vec", c_i, c_vp, c_i, c_ll, c_dp, c_ll, c_d, c_dp, c_d, c_dp)
    f("hb_mat_trans_times_vec", c_i, c_vp, c_i, c_ll, c_dp, c_ll, c_d, c_dp, c_d, c_dp)
    # symdense
    f("hb_mat_times_mat_trans", c_i, c_vp, c_i, c_i, c_ll, c_dp, c_ll, c_dp, c_ll, c_d, c_dp, c_ll, c_d)
    f("hb_mat_add_sub_diagonal", c_i, c_vp, c_dp, c_ll, c_i, c_i, c_d, c_dp, c_i)
    f("hb_mat_add_matrix", c_i, c_vp, c_i, c_i, c_dp, c_ll, c_d, c_dp, c_ll)
    f("hb_mat_copy_rows_from", c_i, c_vp, c_i, c_i, c_dp, c_ll, c_dp, c_ll, c_vp)
    f("hb_mat_copy_block", c_i, c_vp, c_i, c_i, c_dp, c_ll, c_i, c_i, c_dp, c_ll, c_i, c_i)
    f("hb_mat_trans_add_to_sym_upper", c_i, c_vp, c_i, c_i, c_dp, c_ll, c_i, c_i, c_d, c_dp, c_ll)
    f("hb_mat_add_upper_to_sym_upper", c_i, c_vp, c_i, c_dp, c_ll, c_i, c_d, c_dp, c_ll)
    f("hb_lowrank_test_direction", c_i, c_vp, c_dp, c_dp, c_dp, c_dp, c_d, P(c_d))
    f("hb_symdense_create", c_i, c_vp, c_i, P(c_vp))
    f("hb_symdense_destroy", c_i, c_vp)
    f("hb_symdense_matrix", c_vp, c_vp)
    f("hb_symdense_matrix_changed", c_i, c_vp, c_i)
    f("hb_symdense_inertia", c_i, c_vp, P(c_i), P(c_i), P(c_i))
    f("hb_symdense_solve", c_i, c_vp, c_dp, c_i)
    f("hb_symdense_matrix_changed_host", c_i, c_vp, c_vp, c_i)
    f("hb_symdense_solve_host", c_i, c_vp, c_vp, c_i)
    f("hb_debug_diag128_profile", c_i, c_vp, c_i, P(c_ll))
    f("hb_debug_bk_profile", c_i, c_vp, c_i, P(c_ll))
    f("hb_microbench_peak", c_i, c_vp, c_i, P(c_d))
    # lowrank
    f("hb_lowrank_create", c_i, c_vp, c_ll, c_i, c_i, c_i, P(c_vp))
    f("hb_lowrank_destroy", c_i, c_vp)
    f("hb_lowrank_set_patterns", c_i, c_vp, c_dp, c_dp, c_dp, c_dp)
    f("hb_lowrank_set_jacobian", c_i, c_vp, c_dp, c_dp)
    f("hb_lowrank_set_secant", c_i, c_vp, c_i, c_d, c_dp, c_dp, c_vp, c_vp)
    f("hb_lowrank_update", c_i, c_vp, *([c_dp] * 8))
    f("hb_lowrank_condense", c_i, c_vp)
    f("hb_lowrank_condense_async", c_i, c_vp)
    f("hb_lowrank_check", c_i, c_vp)
    f("hb_lowrank_fallback_count", c_i, c_vp)
    f("hb_lowrank_last_condense_chunks", c_i, c_vp)
    f("hb_lowrank_set_condense_mode", c_i, c_vp, c_i)
    f("hb_lowrank_get_condense_mode", c_i, c_vp)
    f("hb_lowrank_solve_compressed", c_i, c_vp, *([c_dp] * 6))
    f("hb_lowrank_compute_directions", c_i, c_vp, P(c_vp), P(c_vp))
    f("hb_lowrank_residual_update", c_i, c_vp, P(c_vp), c_dp, c_dp, c_dp, c_d, c_d, c_dp, c_dp, c_dp, c_dp, c_dp, P(c_vp), P(c_d))
    f("hb_iterate_fraction_to_bdry", c_i, c_vp, P(c_vp), P(c_vp), c_d, P(c_d), P(c_d))
    f("hb_iterate_take_step", c_i, c_vp, P(c_vp), P(c_vp), c_d, c_d, c_i, P(c_vp))
    f("hb_iterate_adjust_duals_plh", c_i, c_vp, P(c_vp), c_d, c_d)
    f("hb_iterate_adjust_small_slacks", c_i, c_vp, P(c_vp), P(c_vp), c_d, c_dp, c_dp, c_dp, c_dp, P(c_i))
    f("hb_iterate_logbar", c_i, c_vp, P(c_vp), c_d, c_d, c_d, c_dp, c_dp, c_dp, P(c_d))
    f("hb_lowrank_lsq_duals", c_i, c_vp, *([c_dp] * 7))
    f("hb_lowrank_secant_reset", c_i, c_vp, c_d, c_i)
    f("hb_lowrank_secant_update", c_i, c_vp, c_dp, c_dp, c_dp, c_dp, c_i, P(c_i))
    f("hb_lowrank_secant_state", c_i, c_vp, P(c_i), P(c_d), P(c_vp), P(c_vp), c_dp, c_dp)
    f("hb_lowrank_compute_directions_w_ir", c_i, c_vp, P(c_vp), P(c_vp), c_d, c_i, P(c_d))
    f("hb_lowrank_kkt_full_times_vec", c_i, c_vp, P(c_vp), P(c_vp))
    f("hb_lowrank_hess_solve", c_i, c_vp, c_dp, c_dp)
    f("hb_lowrank_hess_times_vec", c_i, c_vp, c_d, c_dp, c_d, c_dp, c_i)
    f("hb_lowrank_Dx", c_vp, c_vp)
    f("hb_lowrank_DhInv", c_vp, c_vp)
    f("hb_lowrank_Dd_inv", c_vp, c_vp)
    f("hb_lowrank_N", c_vp, c_vp)
    f("hb_lowrank_last_solve_stats", c_i, c_vp, P(c_i), P(c_d))
    f("hb_lowrank_kkt_system_host", c_i, c_vp, *([c_vp] * 16))
    # mds
    f("hb_mds_create", c_i, c_vp, c_i, c_i, c_i, c_i, P(c_vp))
    f("hb_mds_destroy", c_i, c_vp)
    f("hb_mds_set_sparsity", c_i, c_vp, c_i, c_vp, c_vp, c_i, c_vp, c_vp)
    f("hb_mds_update", c_i, c_vp, *([c_dp] * 6))
    f("hb_mds_build_kkt_matrix", c_i, c_vp, *([c_dp] * 17))
    f("hb_mds_hxs_inertia", c_i, c_vp, P(c_i), P(c_i))
    f("hb_mds_solve_compressed", c_i, c_vp, c_vp, *([c_dp] * 6))
    f("hb_iajaaa_write_matrix_host", c_i, ctypes.c_char_p, c_i, c_dp, c_i, c_i, c_i)
    f("hb_iajaaa_append_vector_host", c_i, ctypes.c_char_p, c_i, c_dp)
    f("hb_iajaaa_write_matrix", c_i, c_vp, ctypes.c_char_p, c_i, c_dp, c_i, c_i, c_i)
    f("hb_iajaaa_append_vector", c_i, c_vp, ctypes.c_char_p, c_i, c_dp)
    f("hb_densekkt_build", c_i, c_vp, c_i, c_i, c_i, c_i, *([c_dp] * 22))
    f("hb_densekkt_solve_compressed", c_i, c_vp, c_vp, c_i, c_i, c_i, c_i, *([c_dp] * 9))
    f("hb_mds_Dx", c_vp, c_vp)
    f("hb_mds_Hxs", c_vp, c_vp)
    f("hb_mds_Dd_inv", c_vp, c_vp)
    _lib = L
    return L


def check(rc: int, what: str = ""):
    if rc != HB_OK:
        raise EngineError(f"{what} failed (code {rc}): {lib().hb_last_error().decode()}")
