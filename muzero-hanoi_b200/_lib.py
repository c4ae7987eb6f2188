"""ctypes binding of libhmz.so (include/hmz.h).  No fallback: if the library is missing or a
call fails, this raises — the product never routes around the CUDA path."""
from __future__ import annotations

import ctypes as C
import os
import threading

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# HMZ_LIB_PATH (tooling): load another build of the library, e.g. an A/B variant produced by tools/build_variant.sh
LIB_PATH = os.environ.get("HMZ_LIB_PATH") or os.path.join(PKG_DIR, "libhmz.so")

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED = 0, -1, -2, -3
FLAG_DONE, FLAG_ILLEGAL, FLAG_GOAL, FLAG_TRUNC = 1, 2, 4, 8
N_ACTIONS, LATENT, HIDDEN, SUPPORT, MAX_DISKS, NO_CHILD = 6, 64, 256, 33, 12, 0xFFFF
LATENT_F32, LATENT_BF16 = 0, 1
SCHEDULE_AUTO, SCHEDULE_PERSISTENT, SCHEDULE_SERVER = 0, 64, 128
MODE_FP32, MODE_BF16, MODE_FP32X3 = 0, 1, 2
REPLAY_NAN, REPLAY_NEGATIVE, REPLAY_SUM, REPLAY_PRIORITY = 1, 2, 4, 8  # status bits of hmz_replay_sample / _set_priorities


class HmzError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libhmz error {code}: {message}")
        self.code = code


class ChildSlot(C.Structure):
    """hmz_child_t — 16 bytes."""

    _fields_ = [("W", C.c_double), ("rwd", C.c_float), ("N", C.c_uint16), ("child", C.c_uint16)]


class NodeHalf(C.Structure):
    """hmz_half_t — 64 bytes."""

    _fields_ = [("c", ChildSlot * 3), ("prior", C.c_float * 3), ("parent", C.c_uint16), ("parent_action", C.c_uint8),
                ("pad", C.c_uint8)]


class NodeRecord(C.Structure):
    """hmz_node_t — 128 bytes."""

    _fields_ = [("h", NodeHalf * 2)]


class SearchDesc(C.Structure):
    """hmz_search_t."""

    _fields_ = [("nodes", C.c_void_p), ("latents", C.c_void_p), ("root_prior", C.c_void_p), ("root_W", C.c_void_p),
                ("minmax", C.c_void_p), ("workspace", C.c_void_p), ("capture", C.c_void_p), ("n_searches", C.c_int64),
                ("n_records", C.c_int32), ("latent_dtype", C.c_int32), ("root_prior_is_f64", C.c_int32), ("schedule", C.c_int32)]


assert C.sizeof(NodeRecord) == 128


class MoveRecord(C.Structure):
    """hmz_move_record_t — 32 bytes."""

    _fields_ = [("root_q", C.c_double), ("state", C.c_uint32), ("reward", C.c_float), ("visits", C.c_uint16 * 6), ("action", C.c_uint8),
                ("flags", C.c_uint8), ("game_lo", C.c_uint16)]


assert C.sizeof(MoveRecord) == 32
RECORD_BYTES = 32
# numpy view of a record buffer (host copy): np.frombuffer(buf, RECORD_DTYPE)
RECORD_DTYPE = [("root_q", "<f8"), ("state", "<u4"), ("reward", "<f4"), ("visits", "<u2", 6), ("action", "u1"), ("flags", "u1"),
                ("game_lo", "<u2")]


class SelfPlayDesc(C.Structure):
    """hmz_selfplay_t."""

    _fields_ = [("search", SearchDesc)] + [(name, C.c_void_p) for name in (
        "weights", "ucb_table", "words", "p0", "v0", "noise", "uniform", "visits", "root_q", "action", "records", "ep_state",
        "ep_action", "ep_flags", "ep_visits", "ep_root_q", "ep_cur_slot", "ep_len", "ep_exp", "pow_table")] + [
        ("discount", C.c_double), ("dirichlet_alpha", C.c_double), ("exploration_eps", C.c_double), ("temperature", C.c_double),
        ("seed", C.c_uint64), ("game_offset", C.c_uint64), ("mode", C.c_int32), ("n_disks", C.c_int32), ("max_steps", C.c_int32),
        ("goal_peg", C.c_int32), ("n_simulations", C.c_int32), ("ep_t_max", C.c_int32), ("reset_word", C.c_uint32),
        ("reserved", C.c_int32)]


class MultiDesc(C.Structure):
    """hmz_multi_t — a heterogeneous search batch: one weight set per 256-search block, one budget per search."""

    _fields_ = [("block_set", C.c_void_p), ("budget", C.c_void_p), ("host_block_budget", C.c_void_p), ("weight_stride", C.c_int64),
                ("n_sets", C.c_int32), ("n_disks", C.c_int32)]


BLOCK = 256  # searches per block of a heterogeneous batch (one weight set each)

_P, _I, _L, _U32, _U64, _D = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64, C.c_double
_SD = C.POINTER(SearchDesc)
_MD = C.POINTER(MultiDesc)

# name -> (restype, argtypes); mirrors include/hmz.h one to one
SIGNATURES = {
    "hmz_last_error": (C.c_char_p, []),
    "hmz_version": (_I, []),
    "hmz_build_flags": (C.c_char_p, []),
    "hmz_launch_count": (_L, []),
    "hmz_device_info": (_I, [C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "hmz_prof_begin": (_I, []),
    "hmz_prof_end": (_I, [_P, _P]),
    "hmz_env_reset": (_I, [_P, _L, _U32, _P]),
    "hmz_env_from_index": (_I, [_P, _P, _L, _I, _P]),
    "hmz_env_to_index": (_I, [_P, _P, _L, _I, _P]),
    "hmz_env_random_reset": (_I, [_P, _L, _I, _I, _U64, _U64, _P]),
    "hmz_env_step": (_I, [_P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _U32, _P]),
    "hmz_env_legal_mask": (_I, [_P, _P, _L, _I, _P]),
    "hmz_env_onehot": (_I, [_P, _P, _L, _I, _P]),
    "hmz_env_solver_distance": (_I, [_P, _P, _L, _I, _I, _P]),
    "hmz_env_step_random": (_I, [_P, _P, _P, _P, _L, _I, _I, _I, _U32, _U64, _U64, _P]),
    "hmz_env_rollout_random": (_I, [_P, _L, _I, _I, _I, _U32, _I, _U64, _U64, _P, _P]),
    "hmz_search_workspace_bytes": (_L, [_L]),
    "hmz_search_minmax_reset": (_I, [_P, _L, _P]),
    "hmz_search_begin": (_I, [_SD, _P, _P]),
    "hmz_search_begin_p0": (_I, [_SD, _P, _P, _D, _P]),
    "hmz_search_select": (_I, [_SD, _I, _P, _D, _P, _P, _P, _P, _I, _P]),
    "hmz_search_child_scores": (_I, [_SD, _P, _P, _P, _D, _P, _P, _P, _P]),
    "hmz_search_expand_backup": (_I, [_SD, _I, _D, _P, _P, _P, _P, _P, _P]),
    "hmz_search_root_policy": (_I, [_SD, _I, _D, _I, _P, _P, _P, _P, _P, _P, _P]),
    "hmz_weights_packed_bytes": (_L, [_I, _I]),
    "hmz_weights_pack": (_I, [C.POINTER(_P), _I, _I, _P]),
    "hmz_net_initial": (_I, [_P, _I, _I, _P, _P, _P, _L, _I, _P, _P, _L, _P]),
    "hmz_net_recurrent": (_I, [_P, _I, _P, _L, _P, _P, _P, _L, _L, _I, _P, _P, _P, _L, _P]),
    "hmz_debug_tc_timeline": (_I, [_P]),
    "hmz_debug_x3_timeline": (_I, [_P]),
    "hmz_debug_persist_stats": (_I, [_P]),
    "hmz_debug_persist_timeline": (_I, [_P]),
    "hmz_debug_gantt": (_I, [_I, _P, _I, _P]),
    "hmz_debug_tree_timeline": (_I, [C.c_longlong, _P]),
    "hmz_debug_div_check": (_I, [_U64, _U64, _P, _P]),
    "hmz_search_run": (_I, [_SD, _P, _I, _I, _P, _D, _P]),
    "hmz_net_initial_multi": (_I, [_P, _MD, _I, _P, _P, _L, _I, _P, _P, _L, _P]),
    "hmz_search_run_multi": (_I, [_SD, _MD, _P, _I, _P, _D, _P]),
    "hmz_search_root_policy_multi": (_I, [_SD, _MD, _D, _I, _P, _P, _P, _P, _P, _P, _P]),
    "hmz_rng_uniform_keyed": (_I, [_P, _L, _U64, _P, _U64, _P, _P]),
    "hmz_rng_dirichlet": (_I, [_P, _L, _D, _U64, _U64, _U64, _P]),
    "hmz_rng_uniform": (_I, [_P, _L, _U64, _U64, _U64, _P]),
    "hmz_debug_philox": (_I, [_P, _P, _I, _P]),
    "hmz_selfplay_move": (_I, [C.POINTER(SelfPlayDesc), _U64, _P]),
    "hmz_learner_param_count": (_L, [_I]),
    "hmz_learner_workspace_bytes": (_L, [_I, _I, _I]),
    "hmz_learner_step": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, C.c_double, C.c_double, C.c_double, C.c_double, _L,
                         _P, _P, _I, _P]),
    "hmz_eval_track": (_I, [_P, _I, _L, _P, _P, _P]),
    "hmz_eval_errors": (_I, [_P, _P, _L, _P, _P]),
    "hmz_episode_record": (_I, [_P, _P, _P, _P, _I, _I, _L, _P, _P, _P, _P, _P, _P, _P]),
    "hmz_episode_close": (_I, [_P, _P, _L, _P, _P, _P]),
    "hmz_episode_ingest": (_I, [_P, _L, _U64, _I, _I, _D, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "hmz_episode_returns": (_I, [_P, _P, _P, _L, _I, _P, _I, _P, _P, _P]),
    "hmz_episode_mc_returns": (_I, [_P, _P, _P, _L, _I, _P, _P, _P, _P]),
    "hmz_episode_rows": (_I, [_P, _P, _L, _L, _I, _P, _P, _P]),
    "hmz_episode_unroll": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _D, _L, _L, _P, _P, _P, _P, _P, _P, _P]),
    "hmz_replay_sample_workspace_bytes": (_L, [_L]),
    "hmz_replay_sample": (_I, [_P, _L, _L, _D, _P, _L, _D, _P, _P, _P, _P, _P]),
    "hmz_replay_set_priorities": (_I, [_P, _L, _P, _P, _L, _P, _P]),
}

_lock = threading.Lock()
_lib = None


def load():
    """Returns the loaded library (ctypes.CDLL) with typed entry points; raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python muzero-hanoi_b200/build.py` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        lenient = bool(os.environ.get("HMZ_LIB_PATH")) and os.environ.get("HMZ_LIB_LENIENT") == "1"  # tooling: older builds
        for name, (restype, argtypes) in SIGNATURES.items():
            if lenient and not hasattr(lib, name):
                continue
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = restype, argtypes
        _lib = lib
    return _lib


def check(rc: int):
    if rc != OK:
        msg = load().hmz_last_error()
        raise HmzError(rc, msg.decode() if msg else "")


def ptr(t):
    """Device (or host) pointer of a torch tensor / numpy array, None -> NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)


def current_stream():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("muzero-hanoi_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
