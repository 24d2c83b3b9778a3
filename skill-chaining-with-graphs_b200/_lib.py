"""ctypes binding of libscg_b200.so (include/scg_b200.h).  No CPU fallback: if the CUDA library is
missing or a call fails, this raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libscg_b200.so")

N_ACTIONS = 5
N_PSI = 6
MAX_OPTIONS = 16
MAX_ORDER = 5
WIN_MAX = 32
GOAL_BIT = 0x80000000
STREAM_ACTION, STREAM_RESET, STREAM_RESELECT, STREAM_TOP = 0, 1, 2, 3


class ScgError(RuntimeError):
    pass


class CtlStruct(C.Structure):
    """struct scg_ctl of include/scg_b200.h: the device-resident controller state."""
    _fields_ = [
        ("n_active", C.c_int32), ("active_mask", C.c_uint32), ("n_promotions", C.c_int32),
        ("last_promotion_step", C.c_uint32), ("manage_calls", C.c_uint32), ("reserved", C.c_uint32 * 3),
        ("parents", C.c_uint32 * MAX_OPTIONS),
    ]


class AgentStruct(C.Structure):
    """struct scg_agent of include/scg_b200.h (field order and types must match)."""
    _fields_ = [
        ("B", C.c_int32), ("K", C.c_int32), ("order", C.c_int32), ("n_active", C.c_int32),
        ("graph", C.c_uint32), ("env_offset", C.c_uint32), ("step", C.c_uint32),
        ("example_capacity", C.c_uint32),
        ("seed", C.c_uint64),
        ("gamma", C.c_float), ("lam", C.c_float), ("epsilon", C.c_float), ("option_bonus", C.c_float),
        ("option_timeout", C.c_int32), ("max_episode_steps", C.c_int32), ("cull", C.c_int32),
        ("carry_valid", C.c_int32),
        ("alpha", C.c_float), ("window_steps", C.c_int32), ("win_cap", C.c_int32), ("win_len", C.c_int32),
        ("ev_cap", C.c_int32), ("ev_len", C.c_int32), ("ring_len", C.c_int32), ("gestation_successes", C.c_int32), ("clf_steps", C.c_int32), ("clf_lr", C.c_float),
        ("top_slots", C.c_int32), ("alpha_top", C.c_float), ("epsilon_top", C.c_float), ("init_horizon", C.c_int32),
        ("merge_overlap", C.c_float), ("goal_x", C.c_float), ("goal_y", C.c_float), ("episode_capacity", C.c_uint32),
        ("x", C.c_void_p), ("y", C.c_void_p), ("vx", C.c_void_p), ("vy", C.c_void_p),
        ("x2", C.c_void_p), ("y2", C.c_void_p), ("vx2", C.c_void_p), ("vy2", C.c_void_p),
        ("action", C.c_void_p), ("option", C.c_void_p), ("t_opt", C.c_void_p), ("ep_steps", C.c_void_p),
        ("start_xy", C.c_void_p), ("start_vxy", C.c_void_p), ("opt_ret", C.c_void_p), ("opt_disc", C.c_void_p),
        ("ep_return", C.c_void_p), ("ep_count", C.c_void_p), ("last_return", C.c_void_p),
        ("reward", C.c_void_p), ("flags", C.c_void_p), ("delta", C.c_void_p), ("q_carry", C.c_void_p),
        ("win_rec", C.c_void_p), ("ev_hist", C.c_void_p), ("ev_pos", C.c_void_p), ("win_top", C.c_void_p), ("trace", C.c_void_p),
        ("W", C.c_void_p), ("Wt", C.c_void_p), ("theta", C.c_void_p), ("dW", C.c_void_p),
        ("cnt", C.c_void_p), ("ctl", C.c_void_p),
        ("ex_xy", C.c_void_p), ("ex_label", C.c_void_p),
        ("ex_count", C.c_void_p), ("n_success", C.c_void_p), ("n_fail", C.c_void_p),
        ("n_success_global", C.c_void_p),
        ("stats", C.c_void_p),
        ("ev_ep", C.c_void_p), ("ep_log", C.c_void_p), ("ep_log_count", C.c_void_p),
        ("option_capacity", C.c_uint32), ("ev_opt", C.c_void_p), ("opt_log", C.c_void_p), ("opt_log_count", C.c_void_p),
        ("traj_n", C.c_uint32), ("traj_env", C.c_void_p), ("traj_capacity", C.c_uint32), ("traj_log", C.c_void_p),
        ("traj_log_count", C.c_void_p), ("traj_len", C.c_int32),
        ("occ_grid", C.c_uint32), ("occ_counts", C.c_void_p), ("occ_len", C.c_int32),
    ]


_P = C.c_void_p
_SIGS = {
    "scg_error_string": (C.c_char_p, [C.c_int]),
    "scg_version": (C.c_int, []),
    "scg_launch_count": (C.c_uint64, []),
    "scg_map_create": (C.c_int, [_P, _P, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, _P, C.c_int,
                                 C.c_int, C.POINTER(_P)]),
    "scg_map_destroy": (C.c_int, [_P]),
    "scg_map_num_edges": (C.c_int, [_P]),
    "scg_map_num_candidates": (C.c_int, [_P]),
    "scg_map_edge_table": (C.c_int, [_P, _P, _P, _P]),
    "scg_map_grid": (C.c_int, [_P, C.POINTER(C.c_int), _P, _P]),
    "scg_step": (C.c_int, [_P, C.c_int] + [_P] * 11 + [C.c_int, _P]),
    "scg_reset": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, C.c_uint64, C.c_uint32, C.c_uint32, _P]),
    "scg_step_host": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P]),
    "scg_features": (C.c_int, [C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "scg_packed_slot_floats": (C.c_int, [C.c_int]),
    "scg_pack_weights": (C.c_int, [C.c_int, C.c_int, _P, _P, _P]),
    "scg_q_eval": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    "scg_select": (C.c_int, [C.c_int, _P, C.c_float, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, _P, _P]),
    "scg_td_error": (C.c_int, [C.c_int, C.c_int, C.c_int] + [_P] * 14 + [C.c_float, _P, _P]),
    "scg_ctx_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(_P)]),
    "scg_ctx_destroy": (C.c_int, [_P]),
    "scg_ctx_set_deterministic": (C.c_int, [_P, C.c_int]),
    "scg_sarsa_update": (C.c_int, [_P, C.c_int] + [_P] * 9 + [C.c_float, _P, _P, _P, _P]),
    "scg_apply": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_float, C.c_float, C.c_int, _P]),
    "scg_clf_eval": (C.c_int, [C.c_int, _P, _P, _P, C.c_int, _P, _P]),
    "scg_clf_decide": (C.c_int, [C.c_int, _P, _P, _P, C.c_int, _P, _P]),
    "scg_clf_grad": (C.c_int, [C.c_int, _P, _P, _P, _P, _P]),
    "scg_clf_fit": (C.c_int, [C.c_int, _P, _P, _P, C.c_int, C.c_float, _P]),
    "scg_agent_step": (C.c_int, [_P, _P, C.POINTER(AgentStruct), _P]),
    "scg_agent_flush": (C.c_int, [_P, C.POINTER(AgentStruct), _P]),
    "scg_agent_ring": (C.c_int, [_P, C.POINTER(AgentStruct), _P]),
    "scg_agent_traj": (C.c_int, [_P, C.POINTER(AgentStruct), _P]),
    "scg_agent_occupancy": (C.c_int, [_P, C.POINTER(AgentStruct), _P]),
    "scg_agent_manage": (C.c_int, [_P, C.POINTER(AgentStruct), _P, _P]),
    "scg_agent_poll": (C.c_int, [_P, C.POINTER(CtlStruct)]),
    "scg_agent_set_ctl": (C.c_int, [_P, C.POINTER(AgentStruct), C.POINTER(CtlStruct), _P]),
    "scg_agent_run": (C.c_int, [_P, _P, C.POINTER(AgentStruct), C.c_int, C.c_int, _P, _P]),
    "scg_agent_sync": (C.c_int, [_P, C.POINTER(AgentStruct), _P, _P]),
    "scg_xchg_create": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(_P)]),
    "scg_xchg_destroy": (C.c_int, [_P]),
    "scg_xchg_handle_bytes": (C.c_int, []),
    "scg_xchg_handle": (C.c_int, [_P, _P]),
    "scg_xchg_connect": (C.c_int, [_P, _P]),
    "scg_xchg_local_ptr": (C.c_int, [_P, C.POINTER(_P)]),
    "scg_xchg_connect_ptrs": (C.c_int, [_P, _P]),
    "scg_xchg_status": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "scg_xchg_set_timeout": (C.c_int, [_P, C.c_double]),
    "scg_xchg_sync": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_float, C.c_float, C.c_int, _P, _P, _P]),
    "scg_agent_step_host": (C.c_int, [_P, _P, C.POINTER(AgentStruct)] + [_P] * 8),
    "scg_agent_run_host": (C.c_int, [_P, _P, C.POINTER(AgentStruct), _P, _P, C.c_int, C.c_int, _P] + [_P] * 6),
    "scg_profile_begin": (C.c_int, [_P, C.c_int, C.c_int]),
    "scg_profile_end": (C.c_int, [_P, _P, _P]),
}

EXPORTS = tuple(_SIGS)
_lib = None


def load():
    """Load the shared library (once).  Raises ScgError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ScgError(f"{LIB_PATH} is missing: run build.sh (or __graft_entry__.build()); "
                       "there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != 0:
        msg = load().scg_error_string(code)
        raise ScgError(f"scg error {code}: {msg.decode() if msg else '?'}")


def ptr(t):
    """Device (or host) pointer of a torch tensor / numpy array, or None."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
