"""ctypes loader for libccx.so (include/ccx.h).  There is no CPU fallback: a missing library, a missing
symbol or a missing CUDA device raises."""
import ctypes
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CCX_LIB_PATH") or os.path.join(PKG, "libccx.so")     # CCX_LIB_PATH: an instrumented build of the same sources (experiments)

i64, i32, u64, u32, f64, vp = (ctypes.c_int64, ctypes.c_int32, ctypes.c_uint64, ctypes.c_uint32,
                               ctypes.c_double, ctypes.c_void_p)

# symbol -> (restype, argtypes); mirrors include/ccx.h one for one
SIGNATURES = {
    "ccx_abi_version": (i32, []),
    "ccx_strerror": (ctypes.c_char_p, [i32]),
    "ccx_last_cuda_error": (ctypes.c_char_p, [vp]),
    "ccx_create": (i32, [i32, ctypes.POINTER(vp)]),
    "ccx_destroy": (i32, [vp]),
    "ccx_set_stream": (i32, [vp, vp]),
    "ccx_synchronize": (i32, [vp]),
    "ccx_launch_count": (i64, [vp]),
    "ccx_graph_replays": (i64, [vp]),
    "ccx_reset": (i32, [vp, i64, vp, i32, u64, i64]),
    "ccx_movegen": (i32, [vp, i64, vp, vp]),
    "ccx_apply": (i32, [vp, i64, vp, vp, vp, vp]),
    "ccx_info": (i32, [vp, i64, vp, vp]),
    "ccx_step_random": (i32, [vp, i64, vp, i64, u64, u32, i32, vp, vp, i64]),
    "ccx_greedy_candidates": (i32, [vp, i64, vp, vp]),
    "ccx_play_greedy": (i32, [vp, i64, vp, i64, u64, i32, vp]),
    "ccx_encode": (i32, [vp, i64, vp, vp, i32]),
    "ccx_mcts_search": (i32, [vp, i64, vp, i32, i32, f64, f64, i32, vp, i32, i32, vp, vp, vp, vp]),
    "ccx_mcts_begin": (i32, [vp, i64, vp, i32, i32, i32, i32]),
    "ccx_mcts_begin_reuse": (i32, [vp, i64, vp, i32, i32, i32, i32, i32, vp, vp, i32, i32, vp]),
    "ccx_mcts_begin_budget": (i32, [vp, i64, vp, i32, i32, i32, i32, vp]),
    "ccx_mcts_set_tiebreak": (i32, [vp, i32, u64, i64]),
    "ccx_mcts_select": (i32, [vp, i64, f64, vp]),
    "ccx_mcts_run_net": (i32, [vp, i64, i32, f64, vp, i32, i32]),
    "ccx_mcts_expand_backup": (i32, [vp, i64, vp, vp, vp, i32, i32]),
    "ccx_mcts_finalize": (i32, [vp, i64, f64, vp, vp, vp, vp]),
    "ccx_mcts_leaf_budget": (i32, [vp, i64, i32, i32]),
    "ccx_mcts_select_leaves": (i32, [vp, i64, i32, f64, vp]),
    "ccx_mcts_expand_backup_leaves": (i32, [vp, i64, i32, vp, vp, vp, i32, i32]),
    "ccx_mcts_run_net_leaves": (i32, [vp, i64, i32, i32, f64, vp, i32, i32]),
    "ccx_mcts_get_root": (i32, [vp, i64, i32, vp, vp, vp, vp, vp]),
    "ccx_mcts_set_root_priors": (i32, [vp, i64, i32, vp]),
    "ccx_mcts_pool_bytes": (i64, [vp]),
    "ccx_mcts_set_gumbel": (i32, [vp, i32, i32, f64, f64, f64, u64]),
    "ccx_mcts_finalize_gumbel": (i32, [vp, i64, vp, vp, vp, vp, vp]),
    "ccx_net_num_weights": (i32, []),
    "ccx_net_load": (i32, [vp, vp, i64]),
    "ccx_net_forward": (i32, [vp, i64, vp, i32, vp, vp]),
    "ccx_softmax_f64": (i32, [vp, i64, vp, vp, vp, vp]),
    "ccx_net_eval": (i32, [vp, i64, vp, vp, vp]),
    "ccx_gamma_noise": (i32, [vp, i64, i32, f64, u64, u32, i64, vp]),
    "ccx_set_slot_ids": (i32, [vp, vp]),
    "ccx_selfplay_advance": (i32, [vp, i64, vp, vp, vp, u64, i32, i64, vp, i64, i32, i32, i32, vp, vp, vp, i32, vp, vp]),
    "ccx_selfplay_finish": (i32, [vp, i64, vp, i32, vp, vp, vp, vp, i32, i32, i32, vp, vp]),
    "ccx_traj_pack": (i32, [vp, i64, vp, vp, vp, vp, vp, vp, vp]),
    "ccx_selfplay_record_pi": (i32, [vp, i64, i32, vp, vp, i32]),
    "ccx_traj_pack_pi": (i32, [vp, i64, vp, vp, vp, vp, vp, vp, vp]),
    "ccx_selfplay_resign": (i32, [vp, i64, vp, u64, i64, vp, f64, i32, f64, vp, vp, vp]),
    "ccx_selfplay_resign_account": (i32, [vp, i64, vp, i32, vp, vp, u64, i64, f64, f64, vp, vp, vp, i64]),
    "ccx_selfplay_playout_cap": (i32, [vp, i64, vp, u64, i64, vp, i32, f64, i32, i32, vp, vp, vp]),
    "ccx_game_advance": (i32, [vp, i64, vp, vp, vp, u64, i64, f64, i32, i32, vp]),
    "ccx_greedy_generate": (i32, [vp, i64, vp, i64, u64, i32, i32, i32, i32, vp, vp, vp, i64, vp, vp, vp, vp]),
    "ccx_cand_to_pi": (i32, [vp, i64, vp, vp]),
    "ccx_net_tc_blob_bytes": (i32, []),
    "ccx_net_tc_num_floats": (i32, []),
    "ccx_net_load_tc": (i32, [vp, vp, i64, vp, i64, i32]),
    "ccx_net_forward_tc": (i32, [vp, i64, vp, vp, vp]),
    "ccx_net_set_mode": (i32, [vp, i32]),
    "ccx_net_set_symmetry": (i32, [vp, i32, u64]),
    "ccx_net_forward_u8": (i32, [vp, i64, vp, vp, vp]),
    "ccx_net_acc_blob_bytes": (i32, []),
    "ccx_net_load_acc": (i32, [vp, vp, i64]),
    "ccx_net_set_acc_contexts": (i32, [vp, i32]),
    "ccx_debug_umma_gemm": (i32, [vp, vp, vp, i32, i32, vp]),
    "ccx_debug_umma_gemm_ts": (i32, [vp, vp, vp, i32, vp]),
    "ccx_debug_umma_gemm_rows": (i32, [vp, vp, i32, i32, vp, i32, i32, vp]),
    "ccx_movegen_host": (i32, [vp, i64, vp, vp]),
    "ccx_apply_host": (i32, [vp, i64, vp, vp, vp, vp]),
    "ccx_step_random_host": (i32, [vp, i64, vp, i64, u64, u32, i32, vp]),
    "ccx_encode_host": (i32, [vp, i64, vp, vp, i32]),
    "ccx_info_host": (i32, [vp, i64, vp, vp]),
    "ccx_greedy_candidates_host": (i32, [vp, i64, vp, vp]),
}

_lib = None


class CcxError(RuntimeError):
    pass


def load():
    """Load libccx.so and bind every symbol of include/ccx.h.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CcxError("libccx.so not built: run `python -m chinesecheckersagent_b200.build` "
                       "(nvcc -gencode arch=compute_100a,code=sm_100a); there is no CPU fallback")
    L = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)          # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if L.ccx_abi_version() != 2:
        raise CcxError("libccx.so ABI version mismatch")
    _lib = L
    return L


def check(L, handle, rc):
    if rc != 0:
        msg = L.ccx_strerror(rc).decode()
        cuda = L.ccx_last_cuda_error(handle).decode() if handle else ""
        raise CcxError("ccx error %d: %s %s" % (rc, msg, cuda))
