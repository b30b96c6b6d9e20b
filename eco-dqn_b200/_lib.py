"""ctypes binding of libecodqn_b200.so (include/ecodqn_b200.h).  No CPU fallback: if the library is missing or a
call fails, this raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ECO_DQN_B200_LIB") or os.path.join(HERE, "lib", "libecodqn_b200.so")   # (override: kernel experiments)

ECO_OK, ECO_ERR_INVALID, ECO_ERR_UNSUPPORTED, ECO_ERR_CUDA, ECO_ERR_STATE = 0, -1, -2, -3, -4
POLICY_ACTIONS, POLICY_NETWORK, POLICY_GREEDY = 0, 1, 2
MPNN_AUTO, MPNN_SIMT, MPNN_TCGEN05 = 0, 1, 2
MPNN_N_PARAMS = 58425
LOSS_MSE, LOSS_HUBER = 0, 1
ENV_IRREVERSIBLE, ENV_DENSE_REWARD = 1, 2      # eco_env_t.reserved mode bits (include/ecodqn_b200.h)
GRAPHS_PM1 = 1                                  # eco_graphs_t.reserved: every coupling in {-1,0,1}
GRAPHS_MIN_CUT = 2                              # eco_graphs_t.reserved: OptimisationTarget.MIN_CUT
MAX_SPINS = 2048
MAX_SPINS_SPARSE = 32768                        # CSR graph sets (eco_sgraphs_t)

vp = C.c_void_p
i32 = C.c_int32


class Graphs(C.Structure):
    _fields_ = [("G", i32), ("N", i32), ("NP", i32), ("reserved", i32),
                ("J", vp), ("gscal", vp), ("deg", vp), ("gstat", vp), ("dmax", vp), ("gain_tab", vp), ("dn_tab", vp),
                ("tc_ops", vp)]


class Episode(C.Structure):
    _fields_ = [("step", i32), ("cut", i32), ("best_cut", i32), ("dist", i32), ("n_improving", i32),
                ("flags", i32), ("n_visited", i32), ("reserved", i32),
                ("score", C.c_double), ("nscore", C.c_double), ("best_score", C.c_double),
                ("best_nscore", C.c_double), ("key", C.c_uint64 * 2), ("total_reward", C.c_double),
                ("last_reward", C.c_double)]


assert C.sizeof(Episode) == 96


class Env(C.Structure):
    _fields_ = [("B", i32), ("N", i32), ("NP", i32), ("NW", i32),
                ("T", i32), ("HCAP", i32), ("use_basin", i32), ("reserved", i32),
                ("basin_reward", C.c_double),
                ("spins", vp), ("hfield", vp), ("last_flip", vp), ("diff_bits", vp), ("graph_idx", vp),
                ("ep", vp), ("visited", vp), ("zobrist", vp), ("tsf_tab", vp), ("imm_tab", vp),
                ("xn", vp), ("xg", vp), ("frac_tab", vp)]


class WGraphs(C.Structure):
    _fields_ = [("G", i32), ("N", i32), ("NP", i32), ("reserved", i32),
                ("J", vp), ("Jf", vp), ("gscal", vp), ("deg", vp), ("gstat", vp), ("dmax", vp)]


class WEnv(C.Structure):
    _fields_ = [("base", Env), ("h", vp), ("cut", vp)]


WGRAPH_NO_DEGREE, WGRAPH_ASYMMETRIC, WGRAPH_NONFINITE = 2, 4, 8   # eco_wgraphs_t.gstat flags


class SGraphs(C.Structure):
    _fields_ = [("G", i32), ("N", i32), ("NP", i32), ("reserved", i32), ("nnz", C.c_int64),
                ("row_ptr", vp), ("col", vp), ("val", vp), ("gscal", vp), ("deg", vp), ("gstat", vp), ("dmax", vp)]


SGRAPH_FIELD_RANGE, SGRAPH_NONCANONICAL = 8, 16                  # eco_sgraphs_t.gstat flags (besides 1, 2, 4)


class Mpnn(C.Structure):
    _fields_ = [("w_init", vp), ("w_edge", vp), ("w_edge_feat", vp), ("w_msg", vp * 3), ("w_upd", vp * 3),
                ("w_pool", vp), ("w_read", vp), ("b_read", vp), ("packed", vp)]


_lib = None


class EcoError(RuntimeError):
    pass


def lib():
    """Load the shared library (once).  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s not found -- run `python __graft_entry__.py` (or eco-dqn_b200/build.py) first; "
                          "this package has no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    P = C.POINTER
    sig = {
        "eco_last_error": (C.c_char_p, []),
        "eco_abi_version": (C.c_int, []),
        "eco_launch_count": (C.c_int64, [C.c_int]),
        "eco_profile_enable": (C.c_int, [C.c_int]),
        "eco_profile_read": (C.c_int, [C.c_int, P(C.c_double), P(C.c_int64)]),
        "eco_graphs_workspace_bytes": (C.c_size_t, [i32, i32]),
        "eco_graphs_bind": (C.c_int, [P(Graphs), vp, i32, i32]),
        "eco_graphs_upload": (C.c_int, [P(Graphs), vp, vp]),
        "eco_graphs_load_dev": (C.c_int, [P(Graphs), vp, vp]),
        "eco_graphs_update": (C.c_int, [P(Graphs), i32, i32, vp, vp]),
        "eco_graphs_load_edges_dev": (C.c_int, [P(Graphs), i32, i32, vp, vp, vp, vp, C.c_int64, i32, vp]),
        "eco_env_workspace_bytes": (C.c_size_t, [i32, i32, i32]),
        "eco_env_bind": (C.c_int, [P(Env), vp, i32, i32, i32, C.c_double]),
        "eco_env_set_tables": (C.c_int, [P(Env), vp, vp, vp, vp]),
        "eco_env_reset": (C.c_int, [P(Graphs), P(Env), vp, vp, vp]),
        "eco_env_step": (C.c_int, [P(Graphs), P(Env), i32, vp, vp, vp, vp, vp, vp, vp]),
        "eco_env_observation": (C.c_int, [P(Env), vp, vp]),
        "eco_env_best_spins": (C.c_int, [P(Env), vp, vp]),
        "eco_env_masked_argmax": (C.c_int, [P(Env), vp, vp, vp]),
        "eco_env_results": (C.c_int, [P(Env), vp, vp, vp, vp]),
        "eco_graph_aggregate": (C.c_int, [P(Graphs), i32, vp, vp, i32, C.c_float, vp, vp]),
        "eco_mpnn_grad_scratch_bytes": (C.c_size_t, [i32, i32]),
        "eco_mpnn_grad": (C.c_int, [P(Graphs), P(Mpnn), i32, vp, vp, vp, C.c_float, vp, vp, i32, vp, vp, vp, vp]),
        "eco_mpnn_grad_ev": (C.c_int, [P(Graphs), P(Mpnn), i32, vp, vp, vp, C.c_float, vp, vp, i32, vp, vp, vp, vp, vp]),
        "eco_mpnn_adam": (C.c_int, [P(Mpnn), vp, vp, vp, i32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, vp]),
        "eco_mpnn_adam_dev": (C.c_int, [P(Mpnn), vp, vp, vp, vp, vp, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, vp]),
        "eco_dqn_masked_td_target": (C.c_int, [i32, i32, i32, vp, vp, vp, vp, vp, C.c_float, i32, i32, vp, vp, vp]),
        "eco_dqn_masked_argmax": (C.c_int, [i32, i32, i32, vp, vp, vp, vp]),
        "eco_dqn_masked_explore": (C.c_int, [P(Env), vp, vp, vp, vp, vp, vp]),
        "eco_mpnn_grad_obs": (C.c_int, [P(Graphs), P(Mpnn), i32, vp, vp, vp, C.c_float, vp, vp, i32, i32, vp, vp, vp, vp, vp]),
        "eco_dp_create": (C.c_int, [P(vp), i32, i32]),
        "eco_dp_handle": (C.c_int, [vp, vp]),
        "eco_dp_open": (C.c_int, [vp, vp]),
        "eco_dp_adam": (C.c_int, [vp, P(Mpnn), vp, vp, vp, vp, vp, C.c_float, C.c_float, C.c_float, C.c_float, vp, vp]),
        "eco_dp_destroy": (None, [vp]),
        "eco_mpnn_scratch_bytes": (C.c_size_t, [i32, i32, i32]),
        "eco_mpnn_packed_bytes": (C.c_size_t, []),
        "eco_mpnn_pack": (C.c_int, [P(Mpnn), vp, vp]),
        "eco_mpnn_forward": (C.c_int, [P(Graphs), P(Mpnn), i32, vp, vp, vp, C.c_float, vp, vp, vp, i32, vp]),
        "eco_rollout": (C.c_int, [P(Graphs), P(Env), P(Mpnn), i32, i32, C.c_float, vp, vp, i32, vp, vp, vp, vp]),
        "eco_wgraphs_workspace_bytes": (C.c_size_t, [i32, i32]),
        "eco_wgraphs_bind": (C.c_int, [P(WGraphs), vp, i32, i32]),
        "eco_wgraphs_load_dev": (C.c_int, [P(WGraphs), vp, vp]),
        "eco_wenv_workspace_bytes": (C.c_size_t, [i32, i32, i32]),
        "eco_wenv_bind": (C.c_int, [P(WEnv), vp, i32, i32, i32, C.c_double]),
        "eco_wenv_reset": (C.c_int, [P(WGraphs), P(WEnv), vp, vp, vp]),
        "eco_wenv_step": (C.c_int, [P(WGraphs), P(WEnv), i32, vp, vp, vp, vp, vp, vp, vp]),
        "eco_wmpnn_forward": (C.c_int, [P(WGraphs), P(Mpnn), i32, vp, vp, vp, C.c_float, vp, vp, vp, i32, vp]),
        "eco_wrollout": (C.c_int, [P(WGraphs), P(WEnv), P(Mpnn), i32, i32, C.c_float, vp, vp, i32, vp, vp, vp, vp]),
        "eco_wenv_results": (C.c_int, [P(WEnv), vp, vp, vp, vp]),
        "eco_sgraphs_workspace_bytes": (C.c_size_t, [i32, i32, C.c_int64]),
        "eco_sgraphs_bind": (C.c_int, [P(SGraphs), vp, i32, i32, C.c_int64]),
        "eco_sgraphs_load_dev": (C.c_int, [P(SGraphs), vp, vp, vp, vp]),
        "eco_senv_workspace_bytes": (C.c_size_t, [i32, i32, i32]),
        "eco_senv_bind": (C.c_int, [P(Env), vp, i32, i32, i32, C.c_double]),
        "eco_senv_reset": (C.c_int, [P(SGraphs), P(Env), vp, vp, vp]),
        "eco_senv_step": (C.c_int, [P(SGraphs), P(Env), i32, vp, vp, vp, vp, vp, vp, vp]),
        "eco_smpnn_scratch_bytes": (C.c_size_t, [i32, i32]),
        "eco_smpnn_forward": (C.c_int, [P(SGraphs), P(Mpnn), i32, vp, vp, vp, C.c_float, vp, vp, vp, vp]),
        "eco_srollout": (C.c_int, [P(SGraphs), P(Env), P(Mpnn), i32, i32, C.c_float, vp, vp, vp, vp, vp, vp]),
        "eco_session_create": (C.c_int, [P(vp), i32, i32, i32, i32, C.c_double, P(vp), i32]),
        "eco_session_destroy": (None, [vp]),
        "eco_session_rollout": (C.c_int, [vp, vp, vp, vp, i32, C.c_float, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)      # AttributeError here means the .so is stale w.r.t. the header
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


EXPORTED = ["eco_last_error", "eco_abi_version", "eco_launch_count", "eco_profile_enable", "eco_profile_read", "eco_graphs_workspace_bytes",
            "eco_graphs_bind", "eco_graphs_upload", "eco_graphs_load_dev", "eco_graphs_update", "eco_graphs_load_edges_dev", "eco_env_workspace_bytes",
            "eco_env_bind", "eco_env_set_tables", "eco_env_reset", "eco_env_step", "eco_env_observation",
            "eco_env_best_spins", "eco_env_masked_argmax", "eco_env_results", "eco_graph_aggregate", "eco_mpnn_grad_scratch_bytes", "eco_mpnn_grad", "eco_mpnn_grad_ev", "eco_mpnn_adam", "eco_mpnn_adam_dev", "eco_dqn_masked_td_target", "eco_dqn_masked_argmax", "eco_dqn_masked_explore", "eco_mpnn_grad_obs", "eco_dp_create", "eco_dp_handle", "eco_dp_open", "eco_dp_adam", "eco_dp_destroy", "eco_mpnn_scratch_bytes", "eco_mpnn_packed_bytes",
            "eco_mpnn_pack", "eco_mpnn_forward", "eco_rollout", "eco_session_create", "eco_session_destroy",
            "eco_session_rollout", "eco_wgraphs_workspace_bytes", "eco_wgraphs_bind", "eco_wgraphs_load_dev",
            "eco_wenv_workspace_bytes", "eco_wenv_bind", "eco_wenv_reset", "eco_wenv_step", "eco_wmpnn_forward", "eco_wrollout",
            "eco_wenv_results", "eco_sgraphs_workspace_bytes", "eco_sgraphs_bind", "eco_sgraphs_load_dev",
            "eco_senv_workspace_bytes", "eco_senv_bind", "eco_senv_reset", "eco_senv_step", "eco_smpnn_scratch_bytes",
            "eco_smpnn_forward", "eco_srollout"]


def check(rc):
    """Map a C return code to the reference's Python error behaviour."""
    if rc == ECO_OK:
        return
    msg = lib().eco_last_error().decode("utf-8", "replace")
    if rc == ECO_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == ECO_ERR_INVALID:
        raise ValueError(msg)
    raise EcoError("libecodqn_b200 error %d: %s" % (rc, msg))
