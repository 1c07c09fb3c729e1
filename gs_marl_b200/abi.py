"""ctypes mirror of include/gsmarl_b200.h and the loader of the sm_100a library.

The product path has no CPU fallback: `load_library()` raises if
`csrc/libgsmarl_b200.so` is missing or does not export every declared symbol.
"""
from __future__ import annotations

import ctypes as C
import os

GSM_ABI_VERSION = 7
GSM_OBS_DIM = 6
GSM_NBR_FEAT_DIM = 6
GSM_MAX_DISCRETE = 16
GSM_MAX_LSA_N = 32
GSM_POLICY_HIDDEN = 64
GSM_POLICY_MAX_ACTIONS = 9
GSM_POLICY_VALUE_HEADS = 2
GSM_POLICY_GAUSS_DIM = 2
GSM_POLICY_GAUSS_N_PARAMS = 1479

GSM_F32, GSM_F64 = 0, 1
GSM_SCN_NAVIGATION, GSM_SCN_POLYGON, GSM_SCN_LINE = 0, 1, 2
GSM_ACT_DISCRETE, GSM_ACT_CONTINUOUS = 0, 1
GSM_ENT_AGENT, GSM_ENT_GOAL, GSM_ENT_OBSTACLE, GSM_ENT_MARKER = 0, 1, 2, 3

_dp = C.POINTER(C.c_double)


class GsmConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("abi_version", C.c_uint32),
        ("dtype", C.c_int32), ("scenario", C.c_int32), ("action_mode", C.c_int32),
        ("n_agents", C.c_int32), ("n_landmarks", C.c_int32), ("max_nbrs", C.c_int32),
        ("episode_length", C.c_int32), ("n_discrete_actions", C.c_int32),
        ("share_reward", C.c_int32), ("cost_obstacles", C.c_int32),
        ("own_goal_always", C.c_int32), ("reserved0", C.c_int32),
        ("dt", C.c_double), ("damping", C.c_double), ("contact_force", C.c_double),
        ("contact_margin", C.c_double), ("sensing_radius", C.c_double),
        ("w_dist", C.c_double), ("w_goal", C.c_double), ("goal_tol", C.c_double),
        ("polygon_radius", C.c_double), ("spawn_extent", C.c_double * 4),
        ("discrete_u", _dp), ("size", _dp), ("collide", C.POINTER(C.c_uint8)),
        ("type", C.POINTER(C.c_int32)), ("mass", _dp), ("accel", _dp), ("max_speed", _dp),
        ("slot_table", _dp),
    ]


class GsmStepIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("obs", C.c_void_p), ("nbr_idx", C.c_void_p),
        ("nbr_feat", C.c_void_p), ("nbr_cnt", C.c_void_p), ("adj", C.c_void_p),
        ("reward", C.c_void_p), ("cost", C.c_void_p), ("done", C.c_void_p),
        ("assign", C.c_void_p),
    ]

    FIELDS = ("actions", "obs", "nbr_idx", "nbr_feat", "nbr_cnt", "adj", "reward", "cost",
              "done", "assign")


class GsmIoSizes(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in
                ("actions", "obs", "nbr_idx", "nbr_feat", "nbr_cnt", "adj", "reward", "cost",
                 "done", "assign", "agent_state", "landmark_pos", "step_count")] + [
        ("adj_words", C.c_int32), ("real_bytes", C.c_int32)]


class GsmPolicyWeights(C.Structure):
    """gsm_policy_weights: row-major [out][in] like torch.nn.Linear.weight, host memory."""
    _H, _A = GSM_POLICY_HIDDEN, GSM_POLICY_MAX_ACTIONS
    _fields_ = [
        ("struct_size", C.c_uint32), ("n_actions", C.c_int32),
        ("ego_w", C.c_float * GSM_OBS_DIM * _H), ("ego_b", C.c_float * _H),
        ("nbr_w", C.c_float * GSM_NBR_FEAT_DIM * _H), ("nbr_b", C.c_float * _H),
        ("att_w", C.c_float * _H), ("att_b", C.c_float),
        ("head_w", C.c_float * (2 * _H) * _A), ("head_b", C.c_float * _A),
        ("value_w", C.c_float * (2 * _H) * GSM_POLICY_VALUE_HEADS), ("value_b", C.c_float * GSM_POLICY_VALUE_HEADS),
    ]


class GsmPolicyIO(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p), ("nbr_feat", C.c_void_p), ("nbr_cnt", C.c_void_p),
        ("actions", C.c_void_p), ("logp", C.c_void_p), ("logits", C.c_void_p),
        ("values", C.c_void_p), ("n_rows", C.c_int64), ("row_offset", C.c_uint64), ("seed", C.c_uint64), ("step", C.c_uint64),
        ("max_nbrs", C.c_int32), ("greedy", C.c_int32),
    ]


class GsmPolicyEvalIO(C.Structure):
    """gsm_policy_eval_io: DEVICE pointers; `params` is the parameters_to_vector(actor) vector."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("n_actions", C.c_int32),
        ("params", C.c_void_p), ("obs", C.c_void_p), ("nbr_feat", C.c_void_p), ("nbr_cnt", C.c_void_p),
        ("actions", C.c_void_p), ("rows", C.c_void_p),
        ("logp", C.c_void_p), ("entropy", C.c_void_p), ("values", C.c_void_p),
        ("n_rows", C.c_int64), ("max_nbrs", C.c_int32), ("reserved", C.c_int32),
    ]


class GsmPolicyGaussWeights(C.Structure):
    """gsm_policy_gauss_weights: the Gaussian actor, row-major [out][in], host memory."""
    _H, _D = GSM_POLICY_HIDDEN, GSM_POLICY_GAUSS_DIM
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("ego_w", C.c_float * GSM_OBS_DIM * _H), ("ego_b", C.c_float * _H),
        ("nbr_w", C.c_float * GSM_NBR_FEAT_DIM * _H), ("nbr_b", C.c_float * _H),
        ("att_w", C.c_float * _H), ("att_b", C.c_float),
        ("mean_w", C.c_float * (2 * _H) * _D), ("mean_b", C.c_float * _D), ("log_std", C.c_float * _D),
        ("value_w", C.c_float * (2 * _H) * GSM_POLICY_VALUE_HEADS), ("value_b", C.c_float * GSM_POLICY_VALUE_HEADS),
    ]


class GsmPolicyGaussIO(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p), ("nbr_feat", C.c_void_p), ("nbr_cnt", C.c_void_p),
        ("actions", C.c_void_p), ("logp", C.c_void_p), ("mean", C.c_void_p),
        ("values", C.c_void_p), ("n_rows", C.c_int64), ("row_offset", C.c_uint64), ("seed", C.c_uint64), ("step", C.c_uint64),
        ("max_nbrs", C.c_int32), ("greedy", C.c_int32),
    ]


class GsmPolicyGaussEvalIO(C.Structure):
    """gsm_policy_gauss_eval_io: DEVICE pointers; `params` is the parameters_to_vector(GaussianGraphActor) vector."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("action_dim", C.c_int32),
        ("params", C.c_void_p), ("obs", C.c_void_p), ("nbr_feat", C.c_void_p), ("nbr_cnt", C.c_void_p),
        ("actions", C.c_void_p), ("rows", C.c_void_p),
        ("logp", C.c_void_p), ("entropy", C.c_void_p), ("values", C.c_void_p),
        ("n_rows", C.c_int64), ("max_nbrs", C.c_int32), ("reserved", C.c_int32),
    ]


GSM_EPISODE_STAT_FIELDS = 16


class GsmEpisodeIO(C.Structure):
    """gsm_episode_io: DEVICE pointers over the buffer's reward / cost / done slots (SPEC.md §13)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("dtype", C.c_int32),
        ("reward", C.c_void_p), ("cost", C.c_void_p), ("done", C.c_void_p),
        ("carry_return", C.c_void_p), ("carry_cost", C.c_void_p), ("carry_length", C.c_void_p),
        ("totals", C.c_void_p), ("episodes", C.c_void_p),
        ("last_return", C.c_void_p), ("last_cost", C.c_void_p), ("last_length", C.c_void_p),
        ("team_last_return", C.c_void_p), ("team_last_cost", C.c_void_p),
        ("n_rows", C.c_int64), ("slot_rows", C.c_int64), ("n_steps", C.c_int32), ("agents_per_env", C.c_int32),
        ("agent_cost_limit", C.c_double), ("team_cost_limit", C.c_double),
    ]


GSM_PPO_STAT_FIELDS = 8


class GsmPpoLossIO(C.Structure):
    """gsm_ppo_loss_io: DEVICE pointers over the buffer's loss inputs and the loss coefficients (SPEC.md §14)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("reserved", C.c_int32),
        ("old_logp", C.c_void_p), ("old_values", C.c_void_p), ("returns", C.c_void_p), ("advantages", C.c_void_p),
        ("adv_moments", C.c_void_p), ("lagrange", C.c_void_p), ("stats", C.c_void_p),
        ("clip", C.c_float), ("value_clip", C.c_float), ("value_coef", C.c_float), ("entropy_coef", C.c_float),
    ]


def policy_n_params(n_actions: int) -> int:
    """GSM_POLICY_N_PARAMS: length of the learner's parameter vector."""
    return 961 + 129 * n_actions + 2 * (2 * GSM_POLICY_HIDDEN + 1)


_H = C.c_void_p  # gsm_env*
_IO = C.POINTER(GsmStepIO)

# name -> (restype, argtypes); every symbol include/gsmarl_b200.h declares.
SYMBOLS = {
    "gsm_abi_version": (C.c_int, []),
    "gsm_status_string": (C.c_char_p, [C.c_int]),
    "gsm_last_error": (C.c_char_p, [_H]),
    "gsm_create": (C.c_int, [C.POINTER(GsmConfig), C.c_int64, C.c_int64, C.c_int, C.POINTER(_H)]),
    "gsm_destroy": (C.c_int, [_H]),
    "gsm_get_io_sizes": (C.c_int, [_H, C.POINTER(GsmIoSizes)]),
    "gsm_reset": (C.c_int, [_H, C.c_uint64, C.c_void_p, C.c_int64, _IO, C.c_void_p]),
    "gsm_step": (C.c_int, [_H, _IO, C.c_void_p]),
    "gsm_rollout": (C.c_int, [_H, C.c_int32, _IO, C.c_void_p]),
    "gsm_set_auto_reset": (C.c_int, [_H, C.c_int]),
    "gsm_set_slot_envs": (C.c_int, [_H, C.c_int64]),
    "gsm_observe": (C.c_int, [_H, _IO, C.c_void_p]),
    "gsm_set_state": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_get_state": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_set_episode": (C.c_int, [_H, C.c_void_p, C.c_void_p]),
    "gsm_get_episode": (C.c_int, [_H, C.c_void_p, C.c_void_p]),
    "gsm_host_io": (C.c_int, [_H, _IO]),
    "gsm_set_host_outputs": (C.c_int, [_H, C.c_uint32, C.c_int32]),
    "gsm_reset_host": (C.c_int, [_H, C.c_uint64, C.c_void_p, C.c_int64, _IO]),
    "gsm_step_host": (C.c_int, [_H, _IO]),
    "gsm_observe_host": (C.c_int, [_H, _IO]),
    "gsm_set_state_host": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_get_state_host": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gsm_kernel_launches": (C.c_int64, [_H]),
    "gsm_lsa": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int,
                          C.c_void_p]),
    "gsm_policy_act": (C.c_int, [C.POINTER(GsmPolicyWeights), C.POINTER(GsmPolicyIO), C.c_int, C.c_void_p]),
    "gsm_policy_last_error": (C.c_char_p, []),
    "gsm_policy_evaluate": (C.c_int, [C.POINTER(GsmPolicyEvalIO), C.c_int, C.c_void_p]),
    "gsm_policy_backward_workspace": (C.c_int64, [C.c_int64, C.c_int32]),
    "gsm_policy_backward": (C.c_int, [C.POINTER(GsmPolicyEvalIO), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gsm_gae": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int64,
                          C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "gsm_collect": (C.c_int, [_H, C.POINTER(GsmPolicyWeights), C.c_int32, _IO, C.c_void_p, C.c_void_p,
                              C.c_uint64, C.c_uint64, C.c_int32, C.c_void_p]),
    "gsm_policy_act_gauss": (C.c_int, [C.POINTER(GsmPolicyGaussWeights), C.POINTER(GsmPolicyGaussIO), C.c_int,
                                       C.c_void_p]),
    "gsm_policy_evaluate_gauss": (C.c_int, [C.POINTER(GsmPolicyGaussEvalIO), C.c_int, C.c_void_p]),
    "gsm_policy_backward_workspace_gauss": (C.c_int64, [C.c_int64]),
    "gsm_policy_backward_gauss": (C.c_int, [C.POINTER(GsmPolicyGaussEvalIO), C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gsm_collect_gauss": (C.c_int, [_H, C.POINTER(GsmPolicyGaussWeights), C.c_int32, _IO, C.c_void_p, C.c_void_p,
                                    C.c_uint64, C.c_uint64, C.c_int32, C.c_void_p]),
    "gsm_ppo_backward_workspace": (C.c_int64, [C.c_int64, C.c_int32]),
    "gsm_ppo_backward_workspace_gauss": (C.c_int64, [C.c_int64]),
    "gsm_ppo_backward": (C.c_int, [C.POINTER(GsmPolicyEvalIO), C.POINTER(GsmPpoLossIO), C.c_void_p, C.c_void_p,
                                   C.c_size_t, C.c_int, C.c_void_p]),
    "gsm_ppo_backward_gauss": (C.c_int, [C.POINTER(GsmPolicyGaussEvalIO), C.POINTER(GsmPpoLossIO), C.c_void_p,
                                         C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gsm_adam_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_int, C.c_void_p]),
    "gsm_episode_stats_workspace": (C.c_int64, [C.c_int64, C.c_int32]),
    "gsm_episode_stats": (C.c_int, [C.POINTER(GsmEpisodeIO), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
}

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libgsmarl_b200.so")
_lib = None


class GsmError(RuntimeError):
    pass


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen the CUDA library and bind every symbol.  Raises — never falls back."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("GSM_LIB_PATH") or LIB_PATH      # GSM_LIB_PATH: A/B builds of the same ABI (profiles/)
    if not os.path.exists(p):
        raise GsmError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback for the product path.")
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise GsmError(f"{p} does not export {name}") from e
        fn.restype, fn.argtypes = res, args
    v = lib.gsm_abi_version()
    if v != GSM_ABI_VERSION:
        raise GsmError(f"ABI mismatch: library {v}, python {GSM_ABI_VERSION}")
    if path is None:
        _lib = lib
    return lib


def check(lib, status: int, handle=None) -> None:
    if status != 0:
        msg = lib.gsm_last_error(handle) or b""
        raise GsmError(f"{lib.gsm_status_string(status).decode()}: {msg.decode()}")
