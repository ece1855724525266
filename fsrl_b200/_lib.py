"""ctypes binding of libfsrl_b200.so (the C-ABI in include/fsrl_b200.h).

There is deliberately NO fallback: if the CUDA library is missing or a symbol is absent the
import fails loudly (a silent CPU path would void every parity claim).
"""
from __future__ import annotations

import ctypes
import os

import torch  # noqa: F401  (loads torch's bundled libnccl/cudart before ours resolve the same SONAMEs)

_HERE = os.path.dirname(os.path.abspath(__file__))
# FSRL_B200_LIB selects another build of the same library (A/B runs of kernel variants); the default is
# the in-tree build
LIB_PATH = os.environ.get("FSRL_B200_LIB") or os.path.join(_HERE, "libfsrl_b200.so")

FSRL_OK, FSRL_EINVAL, FSRL_ECUDA, FSRL_EWORKSPACE = 0, -1, -2, -3


class FsrlCudaError(RuntimeError):
    pass


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (or `make -C fsrl_b200/csrc`). fsrl_b200 has no CPU fallback.")
    return ctypes.CDLL(LIB_PATH)


lib = _load()

c_f32p = ctypes.c_void_p   # device pointers travel as integers
c_u8p = ctypes.c_void_p
c_i32p = ctypes.c_void_p
c_i64 = ctypes.c_int64
c_f64 = ctypes.c_double
c_f32 = ctypes.c_float
c_int = ctypes.c_int
c_size = ctypes.c_size_t
c_vp = ctypes.c_void_p



# ---- C structs of include/fsrl_b200.h -------------------------------------------------------
class Mlp3(ctypes.Structure):
    _fields_ = [("w1t", c_vp), ("b1", c_vp), ("w2t", c_vp), ("b2", c_vp), ("w3t", c_vp),
                ("b3", c_vp), ("in_", c_int), ("H", c_int), ("out", c_int)]


class CollectStats(ctypes.Structure):
    _fields_ = [("step_count", ctypes.c_ulonglong), ("sum_ep_len", ctypes.c_ulonglong),
                ("total_cost", c_f64), ("sum_ep_rew", c_f64), ("episode_count", c_int),
                ("n_episode", c_int), ("n_ready", c_int), ("term_count", c_int),
                ("trunc_count", c_int), ("finished", c_int), ("finished_next", c_int),
                ("pad", c_int)]


class Rollout(ctypes.Structure):
    _fields_ = [("kind", c_int), ("E", c_int), ("max_steps", c_int), ("inline_done", c_int),
                ("seed_env", ctypes.c_uint), ("seed_act", ctypes.c_uint),
                ("env_state", c_vp), ("obs_cur", c_vp), ("env_t", c_vp), ("ep_idx", c_vp),
                ("act_ctr", c_vp), ("active", c_vp), ("done_now", c_vp), ("ep_rew", c_vp),
                ("ep_len", c_vp),
                ("actor", Mlp3), ("log_sigma", c_vp),
                ("head", c_int), ("mode", c_int), ("bounded", c_int), ("action_bound", c_int),
                ("action_scaling", c_int), ("pad0", c_int),
                ("max_action", c_f32), ("expl_sigma", c_f32), ("sigma_min", c_f32),
                ("sigma_max", c_f32), ("tanh_eps", c_f32), ("pad1", c_f32),
                ("act_low", c_f32 * 8), ("act_high", c_f32 * 8),
                ("b_obs", c_vp), ("b_obs_next", c_vp), ("b_act", c_vp), ("b_rew", c_vp),
                ("b_cost", c_vp), ("b_logp", c_vp), ("b_term", c_vp), ("b_trunc", c_vp),
                ("b_ptr", c_vp), ("b_len", c_vp), ("cap", ctypes.c_longlong),
                ("stats", c_vp)]


class PpoUpdate(ctypes.Structure):
    _fields_ = [("theta", c_vp), ("grad", c_vp), ("adam_m", c_vp), ("adam_v", c_vp),
                ("w2n", c_vp), ("scratch", c_vp), ("norm_sq", c_vp), ("stats", c_vp),
                ("mask", c_vp), ("net_off", ctypes.c_longlong * 3),
                ("n_params", ctypes.c_longlong),
                ("n_nets", c_int), ("D", c_int), ("H", c_int), ("A", c_int), ("C", c_int),
                ("actor_out", c_int), ("bmax", c_int), ("head_indep", c_int),
                ("obs", c_vp), ("act", c_vp), ("logp_old", c_vp), ("adv", c_vp), ("ret", c_vp),
                ("values", c_vp), ("ld", ctypes.c_longlong), ("perm", c_vp),
                ("eps_clip", c_f32), ("dual_clip", c_f32), ("vf_coef", c_f32),
                ("max_grad_norm", c_f32), ("max_action", c_f32), ("lagrangian", c_f32),
                ("rescaling", c_f32), ("pad0", c_f32),
                ("bounded", c_int), ("norm_adv", c_int), ("value_clip", c_int),
                ("use_lagrangian", c_int),
                ("lr", c_f64), ("beta1", c_f64), ("beta2", c_f64), ("adam_eps", c_f64),
                ("comm", c_vp), ("moments_w", c_vp), ("moments", c_vp), ("world", c_int),
                ("batch_size", c_int), ("gather", c_vp), ("mb_stats", c_vp), ("barrier", c_vp),
                ("p2p_xg", (c_vp * 8) * 2), ("p2p_flags", c_vp * 8), ("p2p_err", c_vp), ("p2p_part", c_vp),
                ("p2p_rank", c_int), ("p2p_on", c_int),
                ("persist_ws", c_vp), ("persist_ws_floats", ctypes.c_longlong), ("persist_off", c_int), ("pad1", c_int),
                ("p2p_stride", ctypes.c_longlong)]


class NetRef(ctypes.Structure):
    _fields_ = [("off", ctypes.c_longlong), ("w2n_off", ctypes.c_longlong), ("D", c_int), ("H", c_int),
                ("out", c_int), ("n_extra", c_int), ("slot", c_int), ("pad", c_int)]


class NetList(ctypes.Structure):
    _fields_ = [("n", c_int), ("pad", c_int), ("nets", NetRef * 8)]


class Engine(ctypes.Structure):
    _fields_ = [("theta", c_vp), ("grad", c_vp), ("adam_m", c_vp), ("adam_v", c_vp), ("w2n", c_vp),
                ("scratch", c_vp), ("bmax", c_int), ("pad", c_int)]


class EngInput(ctypes.Structure):
    _fields_ = [("xa", c_vp), ("ia", c_vp), ("xb", c_vp), ("ib", c_vp), ("Da", c_int), ("Db", c_int)]


class OffPolicy(ctypes.Structure):
    _fields_ = [("eng", Engine), ("actor", NetList), ("actor_old", NetList), ("critics", NetList),
                ("critics_old", NetList),
                ("algo", c_int), ("D", c_int), ("A", c_int), ("C", c_int), ("twin", c_int),
                ("n_step", c_int), ("bounded", c_int), ("use_alpha", c_int), ("auto_alpha", c_int),
                ("use_lagrangian", c_int), ("seed", ctypes.c_uint), ("pad0", ctypes.c_uint),
                ("gamma", c_f64), ("tau", c_f64), ("critic_lr", c_f64), ("actor_lr", c_f64),
                ("alpha_lr", c_f32), ("target_entropy", c_f32), ("max_action", c_f32),
                ("sigma_min", c_f32), ("sigma_max", c_f32), ("tanh_eps", c_f32), ("lagrangian", c_f32),
                ("rescaling", c_f32),
                ("b_obs", c_vp), ("b_obs_next", c_vp), ("b_act", c_vp), ("b_rew", c_vp), ("b_cost", c_vp),
                ("b_term", c_vp), ("b_trunc", c_vp), ("b_ptr", c_vp), ("b_len", c_vp),
                ("cap", ctypes.c_longlong),
                ("w_term_idx", c_vp), ("w_partial", c_vp), ("w_gpow", c_vp), ("w_vmask", c_vp),
                ("w_target", c_vp), ("w_act_next", c_vp), ("w_logp_next", c_vp), ("w_act", c_vp),
                ("w_logp", c_vp), ("w_keep", c_vp),
                ("actor_out", c_vp), ("actor_old_out", c_vp), ("actor_dout", c_vp),
                ("q_out", c_vp * 4), ("q_dout", c_vp * 4), ("q_dx", c_vp * 4), ("q_old_out", c_vp * 4),
                ("alpha", c_vp), ("alpha_state", c_vp),
                ("comm", c_vp), ("world", c_int), ("pad1", c_int)]


class Cpo(ctypes.Structure):
    _fields_ = [("eng", Engine), ("actor", NetList), ("actor_r", NetList), ("N", ctypes.c_longlong),
                ("ld", ctypes.c_longlong), ("A", c_int), ("bounded", c_int), ("max_action", c_f32),
                ("pad0", c_f32), ("obs", c_vp), ("act", c_vp), ("logp_old", c_vp), ("mean_old", c_vp),
                ("std_old", c_vp), ("adv", c_vp), ("perm", c_vp), ("out", c_vp), ("dout", c_vp),
                ("log_sigma", c_vp)]


ALGO_SAC, ALGO_DDPG = 0, 1
OFF_STATS = 8

MODE_TRAIN, MODE_EVAL, MODE_RANDOM = 0, 1, 2
HEAD_GAUSS_INDEP, HEAD_GAUSS_COND, HEAD_DETERMINISTIC = 0, 1, 2
BOUND_NONE, BOUND_CLIP, BOUND_TANH = 0, 1, 2
PPO_STATS = 8

# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    "fsrl_last_error": (ctypes.c_char_p, []),
    "fsrl_abi_version": (c_int, []),
    "fsrl_abi_sizeof": (c_size, [c_int]),
    "fsrl_sm_count": (c_int, []),
    "fsrl_launch_count": (ctypes.c_ulonglong, []),
    "fsrl_gae_dual_workspace_bytes": (c_size, [c_i64]),
    "fsrl_gae_dual": (c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_u8p, c_u8p, c_f64, c_f64,
                              c_f32p, c_f32p, c_i64, c_i64, c_int, c_vp, c_size, c_vp]),
    "fsrl_env_dims": (c_int, [c_int] + [ctypes.POINTER(c_int)] * 4),
    "fsrl_env_reset_all": (c_int, [ctypes.POINTER(Rollout), c_vp]),
    "fsrl_collect_begin": (c_int, [ctypes.POINTER(Rollout), c_int, c_vp]),
    "fsrl_rollout_steps": (c_int, [ctypes.POINTER(Rollout), c_int, c_vp]),
    "fsrl_mlp_forward": (c_int, [ctypes.POINTER(Mlp3), c_vp, c_vp, ctypes.c_longlong, c_vp, c_vp]),
    "fsrl_engine_slot_floats": (c_size, [c_int, c_int]),
    "fsrl_engine_forward": (c_int, [ctypes.POINTER(Engine), ctypes.POINTER(NetList), ctypes.POINTER(EngInput), c_int, c_int, c_vp]),
    "fsrl_engine_backward": (c_int, [ctypes.POINTER(Engine), ctypes.POINTER(NetList), c_int, c_int, c_vp]),
    "fsrl_engine_wgrad": (c_int, [ctypes.POINTER(Engine), ctypes.POINTER(NetList), ctypes.POINTER(EngInput), c_int, c_int, c_vp, c_vp]),
    "fsrl_engine_adam": (c_int, [ctypes.POINTER(Engine), ctypes.POINTER(NetList), c_f64, c_f64, c_f64, c_f64,
                                 ctypes.c_longlong, c_f64, c_f64, c_vp, c_f64, c_vp]),
    "fsrl_engine_polyak": (c_int, [ctypes.POINTER(Engine), ctypes.POINTER(NetList), ctypes.POINTER(NetList), c_f64, c_vp]),
    "fsrl_engine_sync_mirror": (c_int, [ctypes.POINTER(Engine), ctypes.POINTER(NetList), c_vp]),
    "fsrl_comm_unique_id": (c_int, [ctypes.c_char_p]),
    "fsrl_comm_init": (c_int, [ctypes.c_char_p, c_int, c_int, ctypes.POINTER(c_vp)]),
    "fsrl_comm_destroy": (c_int, [c_vp]),
    "fsrl_allreduce_fused": (c_int, [c_vp, c_vp, ctypes.c_longlong, c_vp]),
    "fsrl_allreduce_ranges": (c_int, [c_vp, c_vp, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_longlong), c_int, c_vp]),
    "fsrl_p2p_stride": (ctypes.c_longlong, [ctypes.c_longlong]),
    "fsrl_p2p_block_bytes": (ctypes.c_longlong, [ctypes.c_longlong]),
    "fsrl_p2p_alloc": (c_int, [ctypes.c_longlong, ctypes.POINTER(c_vp), ctypes.c_char_p]),
    "fsrl_p2p_open": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    "fsrl_p2p_close": (c_int, [c_vp]),
    "fsrl_p2p_free": (c_int, [c_vp]),
    "fsrl_p2p_poll_error": (c_int, [c_vp, ctypes.POINTER(c_int)]),
    "fsrl_allreduce_f64": (c_int, [c_vp, c_vp, ctypes.c_longlong, c_vp]),
    "fsrl_cpo_head": (c_int, [ctypes.POINTER(Cpo), c_int, c_vp, c_vp]),
    "fsrl_focops_head": (c_int, [ctypes.POINTER(Cpo), c_f64, c_f64, c_f64, c_vp, c_vp]),
    "fsrl_cpo_hvp": (c_int, [ctypes.POINTER(Cpo), c_vp, c_vp, c_vp, c_f64, c_vp]),
    "fsrl_cg_solve": (c_int, [ctypes.POINTER(Cpo), c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_longlong, c_int, c_f64, c_f64, c_vp]),
    "fsrl_vec_dot": (c_int, [c_vp, c_vp, ctypes.c_longlong, c_vp, c_vp]),
    "fsrl_vec_axpby": (c_int, [c_f64, c_vp, c_f64, c_vp, ctypes.c_longlong, c_vp]),
    "fsrl_vec_add_scaled": (c_int, [c_vp, c_f64, c_vp, c_vp, ctypes.c_longlong, c_vp]),
    "fsrl_mse_head": (c_int, [c_vp, c_vp, c_vp, ctypes.c_longlong, c_vp, c_vp, c_vp]),
    "fsrl_standardize": (c_int, [c_vp, ctypes.c_longlong, c_vp]),
    "fsrl_engine_wgrad_to": (c_int, [ctypes.POINTER(Engine), ctypes.POINTER(NetList), ctypes.POINTER(EngInput),
                                     ctypes.c_longlong, c_vp, c_vp]),
    "fsrl_nstep_prepare": (c_int, [ctypes.POINTER(OffPolicy), c_vp, c_int, c_vp]),
    "fsrl_offpolicy_steps": (c_int, [ctypes.POINTER(OffPolicy), c_vp, c_int, c_int, ctypes.c_longlong,
                                     ctypes.c_longlong, ctypes.c_ulonglong, c_vp, c_vp]),
    "fsrl_ppo_scratch_floats": (c_size, [c_int, c_int, c_int]),
    "fsrl_ppo_sync_mirror": (c_int, [ctypes.POINTER(PpoUpdate), c_vp]),
    "fsrl_ppo_persist_ws_floats": (c_size, [c_int, c_int, c_int]),
    "fsrl_ppo_persist_p2p_floats": (c_size, [c_int]),
    "fsrl_ppo_persist_active": (c_int, [ctypes.POINTER(PpoUpdate), ctypes.c_longlong, c_int]),
    "fsrl_ppo_lag_epoch": (c_int, [ctypes.POINTER(PpoUpdate), ctypes.c_longlong, c_int, c_int,
                                   ctypes.c_longlong, ctypes.POINTER(c_int), c_vp]),
}


def _bind():
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover - build error
            raise ImportError(f"libfsrl_b200.so lacks symbol {name}; rebuild the library") from e
        fn.restype = res
        fn.argtypes = args


_bind()


def _check_abi_sizes():
    """The ctypes mirrors must have exactly the C sizes (a silent mismatch would let C read
    past the end of a descriptor)."""
    lib.fsrl_abi_sizeof.restype = c_size
    lib.fsrl_abi_sizeof.argtypes = [c_int]
    for which, cls in enumerate((Mlp3, CollectStats, Rollout, PpoUpdate, NetRef, NetList, Engine, EngInput,
                                 OffPolicy, Cpo)):
        want = lib.fsrl_abi_sizeof(which)
        if want != ctypes.sizeof(cls):
            raise ImportError(f"ABI mismatch: {cls.__name__} is {ctypes.sizeof(cls)} bytes in python, "
                              f"{want} in libfsrl_b200.so -- rebuild / update fsrl_b200/_lib.py")


_check_abi_sizes()


def last_error() -> str:
    return lib.fsrl_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Translate a C-ABI return code into the exception the reference would raise."""
    if rc == FSRL_OK:
        return
    msg = last_error()
    if rc == FSRL_EINVAL:
        raise ValueError(msg)
    if rc == FSRL_EWORKSPACE:
        raise MemoryError(msg)
    raise FsrlCudaError(msg)
