"""ctypes binding of libopenrl_b200.so (the C-ABI declared in include/openrl_b200.h).

There is NO fallback: if the library is missing or a symbol is absent the import of the
product path fails loudly (`OrlLibraryError`).  Tensors cross the boundary as raw device
pointers (`tensor.data_ptr()`) plus sizes; calls are asynchronous on the current torch stream.
"""
import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libopenrl_b200.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "openrl_b200.h")


class OrlLibraryError(RuntimeError):
    pass


class OrlError(RuntimeError):
    pass


_c = ctypes
_P = _c.c_void_p
_I = _c.c_int
_D = _c.c_double
_F = _c.c_float
_L = _c.c_longlong

# name -> argtypes  (restype is int unless noted)
_SIGNATURES = {
    "orl_abi_version": [],
    "orl_device_sm_count": [_c.POINTER(_I)],
    "orl_gae": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _D, _D, _I, _P],
}

_lib = None


def declared_symbols():
    """Every function name declared in include/openrl_b200.h."""
    with open(HEADER) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(orl_[a-z0-9_]+)\s*\(", text)))


def load(path=None):
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise OrlLibraryError(
            f"{p} not found: build it with `python -m openrl_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback."
        )
    try:
        lib = ctypes.CDLL(p)
    except OSError as e:  # pragma: no cover
        raise OrlLibraryError(f"cannot load {p}: {e}") from e
    for name, argtypes in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise OrlLibraryError(f"{p} does not export {name}") from e
        fn.argtypes = argtypes
        fn.restype = _I
    lib.orl_last_error.restype = _c.c_char_p
    lib.orl_last_error.argtypes = []
    lib.orl_rnn_workspace_floats.restype = _c.c_int64
    lib.orl_share_workspace_floats.restype = _c.c_int64
    lib.orl_ppo_peer_bucket_bytes.restype = _c.c_int64
    if lib.orl_abi_version() != 1:
        raise OrlLibraryError("ABI version mismatch")
    if path is None:
        _lib = lib
    return lib


def check(code, what=""):
    if code != 0:
        msg = load().orl_last_error().decode(errors="replace")
        raise OrlError(f"{what} failed with code {code}: {msg}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def current_stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


# ---- argument structs (mirror include/openrl_b200.h field for field) -------------------------
class OrlRolloutArgs(ctypes.Structure):
    _fields_ = [
        ("env_kind", _c.c_int32), ("n_envs", _c.c_int32), ("n_agents", _c.c_int32), ("episode_length", _c.c_int32),
        ("t_begin", _c.c_int32), ("t_end", _c.c_int32), ("obs_dim", _c.c_int32), ("critic_obs_dim", _c.c_int32),
        ("n_actions", _c.c_int32), ("activation_id", _c.c_int32), ("deterministic", _c.c_int32),
        ("env_table_len", _c.c_int32),
        ("policy_params", _P), ("policy_obs", _P), ("critic_obs", _P), ("actions", _P), ("action_log_probs", _P),
        ("rewards", _P), ("masks", _P), ("active_masks", _P), ("action_masks", _P), ("exp_noise", _P),
        ("rng_seed", _c.c_uint64), ("rng_step_base", _c.c_uint64), ("rng_counter", _P),
        ("env_f64", _P), ("env_u64", _P), ("env_i32", _P), ("env_table", _P),
        ("ep_return", _P), ("ep_length", _P), ("episode_stats", _P),
        ("head_kind", _c.c_int32), ("rng_row_offset", _c.c_int32),
    ]


class OrlSelfPlayArgs(ctypes.Structure):
    _fields_ = [
        ("rollout", OrlRolloutArgs),
        ("pool_params", _P), ("pool_count", _P), ("pool_stats", _P),
        ("pool_capacity", _c.c_int32), ("pool_stride", _c.c_int32), ("strategy", _c.c_int32), ("reserved", _c.c_int32),
    ]


class OrlPpoArgs(ctypes.Structure):
    _fields_ = [
        ("obs_dim", _c.c_int32), ("critic_obs_dim", _c.c_int32), ("n_actions", _c.c_int32),
        ("activation_id", _c.c_int32), ("flags", _c.c_int32), ("grid_per_net", _c.c_int32),
        ("batch_rows", _c.c_int64), ("row_begin", _c.c_int64), ("total_rows", _c.c_int64),
        ("indices", _P),
        ("policy_obs", _P), ("critic_obs", _P), ("actions", _P), ("old_log_probs", _P), ("advantages", _P),
        ("value_preds", _P), ("returns", _P), ("active_masks", _P), ("action_masks", _P),
        ("gae_stats", _P), ("mb_stats", _P), ("vn_state", _P),
        ("policy_params", _P), ("critic_params", _P),
        ("policy_adam_m", _P), ("policy_adam_v", _P), ("critic_adam_m", _P), ("critic_adam_v", _P),
        ("adam_steps", _P), ("lrs", _P),
        ("clip_param", _F), ("entropy_coef", _F), ("value_loss_coef", _F), ("huber_delta", _F), ("max_grad_norm", _F),
        ("adam_beta1", _F), ("adam_beta2", _F), ("adam_eps", _F), ("weight_decay", _F), ("reserved0", _F),
        ("vn_beta", _D),
        ("partials", _P), ("folded", _P), ("grads", _P), ("train_info", _P),
        ("head_kind", _c.c_int32), ("dual_clip_coeff", _F),
        ("norm_rows", _c.c_int64),
    ]


class OrlPeerArgs(ctypes.Structure):
    """Mirror of OrlPeerArgs (include/openrl_b200.h): the gradient-bucket exchange over NVLink peer memory."""
    _fields_ = [
        ("peer_buffers", _P), ("local_buffer", _P), ("epochs", _P), ("error_flag", _P), ("summed", _P),
        ("world", _c.c_int32), ("rank", _c.c_int32), ("timeout_ms", _c.c_int32), ("reserved", _c.c_int32),
    ]


PEER_MAX_WORLD = 16

_SIGNATURES.update({
    "orl_env_reset": [_I, _I, _I, _P, _P, _P, _P, _I, _c.c_uint64, _P, _P, _P],
    "orl_rollout": [_c.POINTER(OrlRolloutArgs), _P],
    "orl_env_step": [_I, _I, _I, _P, _P, _P, _P, _I, _c.c_uint64, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "orl_critic_values": [_P, _I, _I, _P, _P, _L, _P],
    "orl_selfplay_reset": [_c.POINTER(OrlSelfPlayArgs), _P, _P],
    "orl_selfplay_rollout": [_c.POINTER(OrlSelfPlayArgs), _P],
    "orl_share_param_count": [_I, _I],
    "orl_share_tape_width": [],
    "orl_share_workspace_floats": [_L, _I, _I],
    "orl_share_rollout": [_c.POINTER(OrlRolloutArgs), _P],
    "orl_share_values": [_P, _I, _I, _I, _P, _P, _L, _P],
    "orl_share_fwdbwd": [_c.POINTER(OrlPpoArgs), _P],
    "orl_share_apply": [_c.POINTER(OrlPpoArgs), _P],
    "orl_host_insert": [_P, _I, _I, _I, _P, _P, _P, _P, _P],
    "orl_policy_eval": [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _L, _P],
    "orl_ppo_stride": [_I, _I, _I],
    "orl_ppo_grads_stride": [_I, _I, _I],
    "orl_net_param_count": [_I, _I],
    "orl_ppo_fwdbwd": [_c.POINTER(OrlPpoArgs), _P],
    "orl_ppo_reduce": [_c.POINTER(OrlPpoArgs), _P],
    "orl_ppo_apply": [_c.POINTER(OrlPpoArgs), _P],
    "orl_minibatch_stats": [_P, _c.c_int64, _P, _P, _P, _P],
    "orl_ppo_peer_bucket_bytes": [_I, _I, _I, _I],
    "orl_ppo_reduce_peer": [_c.POINTER(OrlPpoArgs), _c.POINTER(OrlPeerArgs), _P],
    "orl_ppo_apply_peer": [_c.POINTER(OrlPpoArgs), _c.POINTER(OrlPeerArgs), _P],
    "orl_peer_sum_f64": [_c.POINTER(OrlPeerArgs), _I, _P, _I, _P],
})


class OrlRnnArgs(ctypes.Structure):
    """Mirror of OrlRnnArgs (include/openrl_b200.h): recurrent (GRU) rollout / critic / update / optimizer."""
    _fields_ = [
        ("env_kind", _c.c_int32), ("n_envs", _c.c_int32), ("n_agents", _c.c_int32), ("episode_length", _c.c_int32),
        ("t_begin", _c.c_int32), ("t_end", _c.c_int32),
        ("obs_dim", _c.c_int32), ("critic_obs_dim", _c.c_int32), ("n_actions", _c.c_int32), ("activation_id", _c.c_int32),
        ("deterministic", _c.c_int32), ("chunk_length", _c.c_int32),
        ("flags", _c.c_int32), ("env_table_len", _c.c_int32),
        ("n_chunks", _c.c_int64), ("chunk_ids", _P),
        ("policy_params", _P), ("critic_params", _P), ("policy_obs", _P), ("critic_obs", _P),
        ("rnn_states", _P), ("rnn_states_critic", _P),
        ("actions", _P), ("action_log_probs", _P), ("rewards", _P), ("masks", _P), ("active_masks", _P),
        ("value_preds", _P), ("returns", _P), ("advantages", _P), ("exp_noise", _P),
        ("rng_seed", _c.c_uint64), ("rng_step_base", _c.c_uint64), ("rng_counter", _P),
        ("env_f64", _P), ("env_u64", _P), ("env_i32", _P), ("env_table", _P),
        ("ep_return", _P), ("ep_length", _P), ("episode_stats", _P),
        ("gae_stats", _P), ("mb_stats", _P), ("vn_state", _P),
        ("tape", _P), ("grads", _P), ("grads_stride", _c.c_int32), ("reserved1", _c.c_int32),
        ("loss_acc", _P),
        ("policy_adam_m", _P), ("policy_adam_v", _P), ("critic_adam_m", _P), ("critic_adam_v", _P),
        ("adam_steps", _P), ("lrs", _P),
        ("clip_param", _F), ("entropy_coef", _F), ("value_loss_coef", _F), ("huber_delta", _F), ("max_grad_norm", _F),
        ("adam_beta1", _F), ("adam_beta2", _F), ("adam_eps", _F), ("weight_decay", _F), ("dual_clip_coeff", _F),
        ("vn_beta", _D),
        ("train_info", _P),
        ("norm_rows", _c.c_int64),
    ]


_SIGNATURES.update({
    "orl_rnn_param_count": [_I, _I],
    "orl_rnn_tape_width": [],
    "orl_rnn_workspace_floats": [_c.c_int64, _I],
    "orl_rnn_rollout": [_c.POINTER(OrlRnnArgs), _P],
    "orl_rnn_critic": [_c.POINTER(OrlRnnArgs), _P],
    "orl_rnn_fwdbwd": [_c.POINTER(OrlRnnArgs), _P],
    "orl_rnn_apply": [_c.POINTER(OrlRnnArgs), _P],
})

ENV_NONE, ENV_CARTPOLE, ENV_GRIDWORLD, ENV_MPE_SPREAD, ENV_GRIDWORLD_2P = 0, 1, 2, 3, 4
SP_RANDOM, SP_LAST = 0, 1
HEAD_CATEGORICAL, HEAD_GAUSSIAN = 0, 1
GAE_USE_GAE, GAE_PROPER_TIME_LIMITS, GAE_DENORM = 1, 2, 4
PPO_HUBER, PPO_CLIP_VALUE, PPO_VALUE_ACTIVE_MASKS, PPO_POLICY_ACTIVE_MASKS = 1, 2, 4, 8
PPO_VALUENORM, PPO_ADV_NORMALIZE, PPO_MAX_GRAD_NORM, PPO_TENSORCORE = 16, 32, 64, 128
PPO_TF32 = PPO_TENSORCORE   # round-1 name
PPO_A2C, PPO_DUAL_CLIP = 256, 512
PPO_JOINT_ACTION = 1024   # cfg.use_joint_action_loss (JRPO): chunked recurrent update only
