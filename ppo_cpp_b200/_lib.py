"""Loader for libppo_core.so (the C ABI of include/ppo_core.h).

There is no Python/CPU fallback: if the library is missing or does not export a declared symbol the
import fails loudly.  Build it with `python -c "import __graft_entry__ as g; g.build()"` or
`make -C ppo_cpp_b200/csrc`.
"""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
# PPO_CORE_LIB: another build of the same library (A/B measurements of a kernel change on one box)
LIB_PATH = os.environ.get("PPO_CORE_LIB") or os.path.join(HERE, "libppo_core.so")
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "ppo_core.h")

PPO_HOST, PPO_DEVICE = 0, 1
PPO_VF_CLIP_SHARED, PPO_VF_CLIP_NONE, PPO_VF_CLIP_SEPARATE = 0, 1, 2
PPO_ACT_TANH, PPO_ACT_RELU = 0, 1
PPO_ACTION_BOX, PPO_ACTION_DISCRETE = 0, 1
PPO_COMM_ID_BYTES = 128
PPO_IPC_HANDLE_BYTES = 64
ABI_VERSION = 1


class CoreDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int), ("device", C.c_int), ("obs_dim", C.c_int), ("act_dim", C.c_int),
        ("hidden1", C.c_int), ("hidden2", C.c_int), ("n_envs", C.c_int), ("n_steps", C.c_int),
        ("nminibatches", C.c_int), ("noptepochs", C.c_int), ("gamma", C.c_float), ("lam", C.c_float),
        ("ent_coef", C.c_float), ("vf_coef", C.c_float), ("max_grad_norm", C.c_float),
        ("adam_beta1", C.c_float), ("adam_beta2", C.c_float), ("adam_epsilon", C.c_float),
        ("norm_obs", C.c_int), ("norm_reward", C.c_int), ("training", C.c_int),
        ("clip_obs", C.c_float), ("clip_reward", C.c_float), ("norm_gamma", C.c_float), ("norm_epsilon", C.c_float),
        ("seed", C.c_uint64), ("rank", C.c_int), ("world_size", C.c_int), ("env_offset", C.c_int), ("n_envs_global", C.c_int),
    ]


class MetaInfo(C.Structure):
    _fields_ = [
        ("obs_dim", C.c_int), ("act_dim", C.c_int), ("hidden1", C.c_int), ("hidden2", C.c_int),
        ("ent_coef", C.c_float), ("vf_coef", C.c_float), ("max_grad_norm", C.c_float),
        ("adam_beta1", C.c_float), ("adam_beta2", C.c_float), ("adam_epsilon", C.c_float),
        ("n_params_trainable", C.c_int), ("n_params_total", C.c_int),
    ]


class Counters(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("graph_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]


def declared_symbols(header_path: str = HEADER_PATH):
    """Every function the public header declares (used by the CPU test that the .so exports all of them)."""
    with open(header_path) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ppo_[a-z0-9_]+)\s*\(", text)))


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: build the CUDA library first (make -C ppo_cpp_b200/csrc); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    if missing:
        raise ImportError(f"{LIB_PATH} does not export {missing}")
    vp, fp, ip = C.c_void_p, C.c_void_p, C.c_void_p  # float*/int* passed as raw addresses (host or device)
    core = C.c_void_p
    sig = {
        "ppo_last_error": ([], C.c_char_p),
        "ppo_abi_version": ([], C.c_int),
        "ppo_core_desc_default": ([C.POINTER(CoreDesc)], C.c_int),
        "ppo_meta_parse": ([C.c_char_p, C.POINTER(MetaInfo), fp, C.c_size_t], C.c_int),
        "ppo_meta_vf_clip": ([C.c_char_p], C.c_int),
        "ppo_meta_activation": ([C.c_char_p], C.c_int),
        "ppo_meta_action_space": ([C.c_char_p], C.c_int),
        "ppo_core_create": ([C.POINTER(CoreDesc), C.POINTER(core)], C.c_int),
        "ppo_core_create_ex": ([C.POINTER(CoreDesc), C.c_int, C.POINTER(core)], C.c_int),
        "ppo_core_action_space": ([core], C.c_int),
        "ppo_core_destroy": ([core], None),
        "ppo_core_load_meta_txt": ([core, C.c_char_p], C.c_int),
        "ppo_core_set_vf_clip": ([core, C.c_int], C.c_int),
        "ppo_core_vf_clip": ([core], C.c_int),
        "ppo_core_set_activation": ([core, C.c_int], C.c_int),
        "ppo_core_activation": ([core], C.c_int),
        "ppo_core_init_orthogonal": ([core, C.c_uint64], C.c_int),
        "ppo_core_load_checkpoint_data": ([core, C.c_char_p], C.c_int),
        "ppo_core_save_checkpoint_data": ([core, C.c_char_p], C.c_int),
        "ppo_checkpoint_write_index": ([C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.c_size_t], C.c_int),
        "ppo_checkpoint_write_index_ex": ([C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.c_size_t], C.c_int),
        "ppo_core_num_tensors": ([], C.c_int),
        "ppo_core_tensor_name": ([C.c_int], C.c_char_p),
        "ppo_core_tensor_size": ([core, C.c_char_p], C.c_int),
        "ppo_core_get_tensor": ([core, C.c_char_p, fp, C.c_size_t], C.c_int),
        "ppo_core_set_tensor": ([core, C.c_char_p, fp, C.c_size_t], C.c_int),
        "ppo_core_sync": ([core], C.c_int),
        "ppo_core_stream": ([core], vp),
        "ppo_policy_step": ([core, fp, C.c_int, fp, fp, fp, fp, C.c_int], C.c_int),
        "ppo_policy_value": ([core, fp, C.c_int, fp, C.c_int], C.c_int),
        "ppo_policy_mean": ([core, fp, C.c_int, fp, C.c_int], C.c_int),
        "ppo_vecnorm_reset": ([core, fp, fp, C.c_int], C.c_int),
        "ppo_vecnorm_step": ([core, fp, fp, fp, fp, fp, C.c_int], C.c_int),
        "ppo_vecnorm_replay": ([core, fp, fp, fp, C.c_int, fp, fp, C.c_int], C.c_int),
        "ppo_vecnorm_get_stats": ([core, fp, fp, C.POINTER(C.c_double), fp, fp, C.POINTER(C.c_double)], C.c_int),
        "ppo_vecnorm_set_stats": ([core, fp, fp, C.c_double, fp, fp, C.c_double], C.c_int),
        "ppo_vecnorm_set_training": ([core, C.c_int], C.c_int),
        "ppo_running_stats_update": ([core, fp, fp, C.POINTER(C.c_double), C.c_int, fp, C.c_int, C.c_int], C.c_int),
        "ppo_matrix_clamp": ([core, fp, C.c_size_t, C.c_float, C.c_float, fp, C.c_int], C.c_int),
        "ppo_gae": ([core, fp, fp, fp, fp, fp, C.c_int, C.c_int, C.c_float, C.c_float, fp, fp, C.c_int], C.c_int),
        "ppo_runner_reset": ([core, fp, C.c_int], C.c_int),
        "ppo_runner_act": ([core, C.c_int, fp, C.c_int], C.c_int),
        "ppo_runner_observe": ([core, C.c_int, fp, fp, fp, C.c_int], C.c_int),
        "ppo_runner_finish": ([core], C.c_int),
        "ppo_runner_rollout_host": ([core, C.c_void_p, C.c_void_p, fp], C.c_int),
        "ppo_runner_rollout_replay": ([core, fp, fp, fp, fp], C.c_int),
        "ppo_synth_env_reset": ([core], C.c_int),
        "ppo_rollout_synthetic": ([core], C.c_int),
        "ppo_rollout_get": ([core, C.c_char_p, fp, C.c_size_t], C.c_int),
        "ppo_rollout_set": ([core, C.c_char_p, fp, C.c_size_t], C.c_int),
        "ppo_shuffle_seed": ([core, C.c_uint], C.c_int),
        "ppo_host_srand_rand": ([C.c_uint, C.c_int, ip], C.c_int),
        "ppo_host_random_shuffle": ([C.c_uint, C.c_int, C.c_int, ip], C.c_int),
        "ppo_train_update": ([core, C.c_float, C.c_float, fp], C.c_int),
        "ppo_train_update_vf": ([core, C.c_float, C.c_float, C.c_float, fp], C.c_int),
        "ppo_train_set_permutation": ([core, ip, C.c_int], C.c_int),
        "ppo_train_get_permutation": ([core, C.c_int, ip, C.c_int], C.c_int),
        "ppo_train_minibatch": ([core, C.c_int, C.c_float, C.c_float, fp, fp], C.c_int),
        "ppo_train_minibatch_vf": ([core, C.c_int, C.c_float, C.c_float, C.c_float, fp, fp], C.c_int),
        "ppo_advnorm": ([core, fp, fp, C.c_int, fp], C.c_int),
        "ppo_loss_grad": ([core, fp, fp, fp, fp, fp, fp, C.c_int, C.c_float, fp, fp], C.c_int),
        "ppo_loss_grad_vf": ([core, fp, fp, fp, fp, fp, fp, C.c_int, C.c_float, C.c_float, fp, fp], C.c_int),
        "ppo_learn_update_synthetic": ([core, C.c_float, C.c_float, fp], C.c_int),
        "ppo_comm_get_unique_id": ([C.c_char_p], C.c_int),
        "ppo_comm_init": ([core, C.c_char_p, C.c_int, C.c_int], C.c_int),
        "ppo_comm_ipc_handle": ([core, C.c_char_p], C.c_int),
        "ppo_comm_ipc_open": ([core, C.c_char_p, C.c_int], C.c_int),
        "ppo_comm_error": ([core], C.c_int),
        "ppo_comm_set_p2p": ([core, C.c_int], C.c_int),
        "ppo_core_counters": ([core, C.POINTER(Counters), C.c_int], C.c_int),
        "ppo_core_graph_builds": ([core, C.POINTER(C.c_uint64)], C.c_int),
        "ppo_core_kernel_family": ([core, C.c_char_p], C.c_char_p),
        "ppo_profile_kernel": ([core, C.c_char_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int)], C.c_int),
    }
    undeclared = [s for s in declared_symbols() if s not in sig]
    if undeclared:
        raise ImportError(f"ctypes signatures missing for {undeclared}")
    for name, (args, res) in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = res
    if lib.ppo_abi_version() != ABI_VERSION:
        raise ImportError(f"libppo_core.so ABI {lib.ppo_abi_version()} != binding ABI {ABI_VERSION}")
    _lib = lib
    return lib
