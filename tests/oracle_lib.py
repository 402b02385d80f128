"""ctypes binding of the CPU oracle (oracle/libppo_oracle.so).  TEST INFRASTRUCTURE ONLY.

Imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs.
Nothing under ppo_cpp_b200/ may import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")

f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")


class Dims(C.Structure):
    _fields_ = [("obs_dim", C.c_int), ("act_dim", C.c_int), ("h1", C.c_int), ("h2", C.c_int)]


class HParams(C.Structure):
    _fields_ = [("ent_coef", C.c_float), ("vf_coef", C.c_float), ("clip_norm", C.c_float),
                ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float)]


class GlibcRand(C.Structure):
    _fields_ = [("ring", C.c_uint32 * 31), ("fi", C.c_int), ("ri", C.c_int)]


class RStats(C.Structure):
    _fields_ = [("dim", C.c_int), ("mean", C.POINTER(C.c_float)), ("var", C.POINTER(C.c_float)), ("count", C.c_double)]


class VecNorm(C.Structure):
    _fields_ = [("n_envs", C.c_int), ("obs_dim", C.c_int), ("training", C.c_int), ("norm_obs", C.c_int),
                ("norm_reward", C.c_int), ("clip_obs", C.c_float), ("clip_reward", C.c_float), ("gamma", C.c_float),
                ("epsilon", C.c_float), ("obs_rms", RStats), ("ret_rms", RStats), ("ret", C.POINTER(C.c_float))]


class LearnerDesc(C.Structure):
    _fields_ = [("dims", Dims), ("hp", HParams), ("n_envs", C.c_int), ("n_steps", C.c_int),
                ("nminibatches", C.c_int), ("noptepochs", C.c_int), ("gamma", C.c_float), ("lam", C.c_float),
                ("lr", C.c_float), ("cliprange", C.c_float), ("seed", C.c_uint64), ("shuffle_seed", C.c_uint),
                ("env_kind", C.c_int), ("threads", C.c_int)]


def build(fast: bool = False, native_dir: str = None) -> str:
    """Path of the oracle library: the exact build in oracle/, or the -march=native fast build compiled into `native_dir`."""
    if not fast:
        subprocess.run(["make", "-s", "-C", ORACLE_DIR, "exact"], check=True)
        return os.path.join(ORACLE_DIR, "libppo_oracle.so")
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "fast", f"NATIVE_DIR={native_dir}"], check=True)
    return os.path.join(native_dir, "libppo_oracle_fast.so")


_libs = {}


def load(fast: bool = False):
    if fast in _libs:
        return _libs[fast]
    if fast:
        # built for the host that runs it, outside the tree (bench.py must work from a read-only checkout); the directory
        # can go once the library is mapped
        with tempfile.TemporaryDirectory(prefix="ppo_oracle_fast_") as d:
            lib = C.CDLL(build(True, d))
    else:
        lib = C.CDLL(build())
    vp = C.c_void_p
    lib.oracle_param_offset.argtypes = [C.POINTER(Dims), C.c_int]
    lib.oracle_param_offset.restype = C.c_int
    lib.oracle_philox4x32_10.argtypes = [u32p, u32p, u32p]
    lib.oracle_normal_eps.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, f32p]
    lib.oracle_u32_to_unit_float.argtypes = [C.c_uint32]
    lib.oracle_u32_to_unit_float.restype = C.c_float
    lib.oracle_srand.argtypes = [C.POINTER(GlibcRand), C.c_uint]
    lib.oracle_rand.argtypes = [C.POINTER(GlibcRand)]
    lib.oracle_rand.restype = C.c_int
    lib.oracle_random_shuffle.argtypes = [C.POINTER(GlibcRand), i32p, C.c_int]
    lib.oracle_perm_to_gather.argtypes = [i32p, C.c_int, i32p]
    for suf, rp in (("f32", f32p), ("f64", f64p)):
        getattr(lib, f"oracle_policy_step_{suf}").argtypes = [C.POINTER(Dims), f32p, f32p, C.c_int, vp, vp, vp, vp, vp]
        real = C.c_float if suf == "f32" else C.c_double
        getattr(lib, f"oracle_gae_{suf}").argtypes = [f32p, f32p, f32p, f32p, f32p, C.c_int, C.c_int, real, real, rp, rp]
        getattr(lib, f"oracle_advnorm_{suf}").argtypes = [f32p, f32p, C.c_int, rp]
        getattr(lib, f"oracle_loss_grad_{suf}").argtypes = [C.POINTER(Dims), C.POINTER(HParams), f32p, f32p, f32p, rp, f32p,
                                                           f32p, f32p, C.c_int, real, rp, rp]
        fn = getattr(lib, f"oracle_clip_adam_{suf}")
        fn.argtypes = [C.POINTER(HParams), C.c_int, real, rp, rp, rp, rp, C.POINTER(real), C.POINTER(real)]
        fn.restype = real
    lib.oracle_rstats_update_f32.argtypes = [C.POINTER(RStats), f32p, C.c_int]
    lib.oracle_rstats_update_f64.argtypes = [f64p, f64p, C.POINTER(C.c_double), C.c_int, f64p, C.c_int]
    lib.oracle_vecnorm_create.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.oracle_vecnorm_create.restype = C.POINTER(VecNorm)
    lib.oracle_vecnorm_destroy.argtypes = [C.POINTER(VecNorm)]
    lib.oracle_vecnorm_reset_f32.argtypes = [C.POINTER(VecNorm), f32p, f32p]
    lib.oracle_vecnorm_step_f32.argtypes = [C.POINTER(VecNorm), f32p, f32p, f32p, f32p, f32p]
    lib.oracle_matrix_clamp_f32.argtypes = [f32p, C.c_int, C.c_float, C.c_float, f32p]
    lib.oracle_synth_env_create.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_uint32]
    lib.oracle_synth_env_create.restype = vp
    lib.oracle_synth_env_destroy.argtypes = [vp]
    lib.oracle_synth_env_reset.argtypes = [vp, f32p]
    lib.oracle_synth_env_step.argtypes = [vp, f32p, f32p, f32p, f32p]
    lib.oracle_learner_create.argtypes = [C.POINTER(LearnerDesc), f32p]
    lib.oracle_learner_create.restype = vp
    lib.oracle_learner_destroy.argtypes = [vp]
    lib.oracle_learner_rollout.argtypes = [vp]
    lib.oracle_learner_train.argtypes = [vp, f32p]
    lib.oracle_learner_buffer.argtypes = [vp, C.c_int]
    lib.oracle_learner_buffer.restype = C.POINTER(C.c_float)
    lib.oracle_learner_params.argtypes = [vp]
    lib.oracle_learner_params.restype = C.POINTER(C.c_float)
    lib.oracle_learner_threads.argtypes = [vp]
    lib.oracle_learner_threads.restype = C.c_int
    lib.oracle_learner_get_norm.argtypes = [vp, f32p, f32p, C.POINTER(C.c_double), C.POINTER(C.c_float),
                                            C.POINTER(C.c_float), C.POINTER(C.c_double)]
    _libs[fast] = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Oracle:
    """Convenience wrapper with numpy in / numpy out."""

    def __init__(self, obs_dim=18, act_dim=18, h1=4, h2=5, ent_coef=0.0007160293171182275, vf_coef=0.5,
                 clip_norm=0.5, beta1=0.9, beta2=0.999, adam_eps=1e-5, fast=False):
        self.lib = load(fast)
        self.dims = Dims(obs_dim, act_dim, h1, h2)
        self.hp = HParams(ent_coef, vf_coef, clip_norm, beta1, beta2, adam_eps)
        self.P = self.lib.oracle_param_offset(C.byref(self.dims), 13)
        self.Pq = self.lib.oracle_param_offset(C.byref(self.dims), 15)

    def offset(self, t):
        return self.lib.oracle_param_offset(C.byref(self.dims), t)

    def policy_step(self, params, obs, eps=None, prec="f64"):
        n = obs.shape[0]
        dt = np.float32 if prec == "f32" else np.float64
        A = self.dims.act_dim
        action, mean = np.zeros((n, A), dt), np.zeros((n, A), dt)
        value, nlp = np.zeros(n, dt), np.zeros(n, dt)
        epsc = None if eps is None else np.ascontiguousarray(eps, np.float32)
        getattr(self.lib, f"oracle_policy_step_{prec}")(C.byref(self.dims), np.ascontiguousarray(params, np.float32),
                                                        np.ascontiguousarray(obs, np.float32), n, _ptr(epsc), _ptr(action),
                                                        _ptr(value), _ptr(nlp), _ptr(mean))
        return action, value, nlp, mean

    def gae(self, rewards, values, dones, last_values, last_dones, gamma, lam, prec="f64"):
        T, N = rewards.shape
        dt = np.float32 if prec == "f32" else np.float64
        advs, rets = np.zeros((T, N), dt), np.zeros((T, N), dt)
        c = lambda a: np.ascontiguousarray(a, np.float32)
        getattr(self.lib, f"oracle_gae_{prec}")(c(rewards), c(values), c(dones), c(last_values), c(last_dones), T, N,
                                                gamma, lam, advs, rets)
        return advs, rets

    def advnorm(self, returns, values, prec="f64"):
        n = returns.shape[0]
        out = np.zeros(n, np.float32 if prec == "f32" else np.float64)
        getattr(self.lib, f"oracle_advnorm_{prec}")(np.ascontiguousarray(returns, np.float32),
                                                    np.ascontiguousarray(values, np.float32), n, out)
        return out

    def loss_grad(self, params, obs, actions, advs, returns, old_nlp, old_v, cliprange, prec="f64"):
        B = obs.shape[0]
        dt = np.float32 if prec == "f32" else np.float64
        grads, losses = np.zeros(self.P, dt), np.zeros(5, dt)
        c = lambda a: np.ascontiguousarray(a, np.float32)
        getattr(self.lib, f"oracle_loss_grad_{prec}")(C.byref(self.dims), C.byref(self.hp), c(params), c(obs), c(actions),
                                                      np.ascontiguousarray(advs, dt), c(returns), c(old_nlp), c(old_v), B,
                                                      cliprange, grads, losses)
        return grads, losses

    def clip_adam(self, lr, params, m, v, grads, b1p, b2p, prec="f64"):
        dt = np.float32 if prec == "f32" else np.float64
        real = C.c_float if prec == "f32" else C.c_double
        p, mm, vv, g = (np.array(a, dt, copy=True) for a in (params, m, v, grads))
        b1, b2 = real(b1p), real(b2p)
        gn = getattr(self.lib, f"oracle_clip_adam_{prec}")(C.byref(self.hp), p.size, lr, p, mm, vv, g, C.byref(b1), C.byref(b2))
        return p, mm, vv, g, b1.value, b2.value, gn


def glibc_shuffle(seed: int, n: int, epochs: int = 1):
    """Permutation index arrays after each of `epochs` compounded std::random_shuffle calls (oracle restatement)."""
    lib = load()
    st = GlibcRand()
    lib.oracle_srand(C.byref(st), seed)
    perm = np.arange(n, dtype=np.int32)
    out = []
    for _ in range(epochs):
        lib.oracle_random_shuffle(C.byref(st), perm, n)
        out.append(perm.copy())
    return out
