"""Thin Python mirror of the C ABI (include/ppo_core.h) used by the tests and bench.py.

numpy arrays go through the PPO_HOST path of the library (host pointers, copies inside the call);
torch CUDA tensors (anything with .data_ptr() and .is_cuda) go through PPO_DEVICE.  All compute is
in libppo_core.so — this module holds no arithmetic.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib
from ._lib import PPO_DEVICE, PPO_HOST, CoreDesc, Counters, MetaInfo

LOSS_NAMES = ("pg_loss", "vf_loss", "entropy", "approxkl", "clipfrac")
# the value losses of ppo_vf_clip (include/ppo_core.h), by the names write_meta_txt(vf_clip=...) takes
VF_CLIP_MODES = {"shared": _lib.PPO_VF_CLIP_SHARED, "none": _lib.PPO_VF_CLIP_NONE, "separate": _lib.PPO_VF_CLIP_SEPARATE}
VF_CLIP_NAMES = {v: k for k, v in VF_CLIP_MODES.items()}
# the hidden-layer activations of ppo_activation, by the names write_meta_txt(activation=...) takes
ACTIVATIONS = {"tanh": _lib.PPO_ACT_TANH, "relu": _lib.PPO_ACT_RELU}
ACTIVATION_NAMES = {v: k for k, v in ACTIVATIONS.items()}
# the policy heads of ppo_action_space, by the names write_meta_txt(action_space=...) takes
ACTION_SPACES = {"box": _lib.PPO_ACTION_BOX, "discrete": _lib.PPO_ACTION_DISCRETE, "multi_discrete": _lib.PPO_ACTION_MULTI_DISCRETE,
                 "multi_binary": _lib.PPO_ACTION_MULTI_BINARY}
ACTION_SPACE_NAMES = {v: k for k, v in ACTION_SPACES.items()}
# the rollout buffers every core has (a masking core adds "action_masks", [n_batch, act_dim])
BUFFER_WIDTH = {"obs": None, "returns": 1, "dones": 1, "actions": None, "values": 1, "neglogpacs": 1,
                "true_rewards": 1, "unnormalized_rewards": 1}


class PPOError(RuntimeError):
    pass


def _check(lib, status):
    if status != 0:
        raise PPOError(f"[{status}] {lib.ppo_last_error().decode()}")


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _addr(a):
    if a is None:
        return None
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    return a.ctypes.data


def _is_dev(a):
    return hasattr(a, "is_cuda") and a.is_cuda


def _mask(m, n, width):
    """An action mask (bool or 0 / 1 values, [n, width]) as the uint8 array the C ABI takes.  A mask of another shape, or with a value
    that is not an integer 0 .. 255, is a ValueError here (the library would read past the array, or see the value rounded); the
    other integers go through unchanged, so that the library reports them with its row and column."""
    if m is None:
        return None
    a = np.asarray(m)
    if a.shape != (n, width):
        raise ValueError(f"an action mask has shape ({n}, {width}) (one entry per logit), not {a.shape}")
    if a.dtype != np.uint8:
        f = a.astype(np.float64)
        bad = ~np.isfinite(f) | (f != np.round(f)) | (f < 0) | (f > 255)
        if bad.any():
            r, j = (int(x) for x in np.argwhere(bad)[0])
            raise ValueError(f"action mask row {r}, column {j} is {a[r, j]}: a mask entry is 1 (allowed) or 0 (forbidden)")
    return np.ascontiguousarray(a, np.uint8)


def meta_parse(path: str):
    lib = _lib.load()
    info = MetaInfo()
    _check(lib, lib.ppo_meta_parse(path.encode(), C.byref(info), None, 0))
    params = np.zeros(info.n_params_total, np.float32)
    _check(lib, lib.ppo_meta_parse(path.encode(), C.byref(info), params.ctypes.data, params.size))
    return info, params


def meta_vf_clip(path: str) -> str:
    """Which value loss the graph file builds: "shared", "none" or "separate" (read by the C parser)."""
    lib = _lib.load()
    r = lib.ppo_meta_vf_clip(path.encode())
    if r < 0:
        _check(lib, r)
    return VF_CLIP_NAMES[r]


def meta_activation(path: str) -> str:
    """The hidden-layer activation of the graph file's forward pass: "tanh" or "relu" (read by the C parser)."""
    lib = _lib.load()
    r = lib.ppo_meta_activation(path.encode())
    if r < 0:
        _check(lib, r)
    return ACTIVATION_NAMES[r]


def meta_action_space(path: str) -> str:
    """The action space of the graph file's policy head: "box" (Gaussian, model/pi/logstd) or "discrete" (categorical, read by the
    C parser)."""
    lib = _lib.load()
    r = lib.ppo_meta_action_space(path.encode())
    if r < 0:
        _check(lib, r)
    return ACTION_SPACE_NAMES[r]


def _nvec(fn, *args) -> list:
    n = fn(*args, None, 0)
    if n < 0:
        return n
    out = np.zeros(n, np.int32)
    r = fn(*args, out.ctypes.data, n)
    return r if r < 0 else [int(x) for x in out]


def meta_action_nvec(path: str) -> list:
    """The choices per action column of the graph file's head (read by the C parser): [n] for "discrete", nvec for "multi_discrete",
    2s for "multi_binary"; PPOError for "box"."""
    lib = _lib.load()
    r = _nvec(lib.ppo_meta_action_nvec, path.encode())
    if isinstance(r, int):
        _check(lib, r)
    return r


def host_rand(seed: int, count: int) -> np.ndarray:
    lib = _lib.load()
    out = np.zeros(count, np.int32)
    _check(lib, lib.ppo_host_srand_rand(seed, count, out.ctypes.data))
    return out


def host_random_shuffle(seed: int, n: int, epochs: int) -> np.ndarray:
    lib = _lib.load()
    out = np.zeros((epochs, n), np.int32)
    _check(lib, lib.ppo_host_random_shuffle(seed, n, epochs, out.ctypes.data))
    return out


def comm_unique_id() -> bytes:
    lib = _lib.load()
    buf = C.create_string_buffer(_lib.PPO_COMM_ID_BYTES)
    _check(lib, lib.ppo_comm_get_unique_id(buf))
    return buf.raw


class PPOCore:
    def __init__(self, activation: str = "tanh", action_space: str = "box", nvec=None, **kw):
        self.lib = _lib.load()
        if activation not in ACTIVATIONS:
            raise ValueError(f"activation must be one of {sorted(ACTIVATIONS)}, not {activation!r}")
        if action_space not in ACTION_SPACES:
            raise ValueError(f"action_space must be one of {sorted(ACTION_SPACES)}, not {action_space!r}")
        if (action_space == "multi_discrete") != (nvec is not None):
            raise ValueError("nvec goes with action_space='multi_discrete' (and only with it)")
        if nvec is not None:
            kw.setdefault("act_dim", int(sum(nvec)))  # the logits of the k slices
        d = CoreDesc()
        _check(self.lib, self.lib.ppo_core_desc_default(C.byref(d)))
        for k, v in kw.items():
            if not hasattr(d, k):
                raise TypeError(f"unknown ppo_core_desc field {k}")
            setattr(d, k, v)
        self.desc = d
        self._h = C.c_void_p()
        if action_space == "box":
            _check(self.lib, self.lib.ppo_core_create(C.byref(d), C.byref(self._h)))
        elif nvec is not None:
            nv = np.ascontiguousarray(nvec, np.int32)
            _check(self.lib, self.lib.ppo_core_create_nvec(C.byref(d), nv.ctypes.data, nv.size, C.byref(self._h)))
        else:
            _check(self.lib, self.lib.ppo_core_create_ex(C.byref(d), ACTION_SPACES[action_space], C.byref(self._h)))
        self.O, self.A = d.obs_dim, d.act_dim
        # floats of one stored action: the action vector (Box), the index of a categorical head (Discrete), one index per slice
        # (MultiDiscrete), one bit per logit (MultiBinary)
        self.AW = d.act_dim if action_space == "box" else len(self.nvec)
        self.n_envs, self.n_steps = d.n_envs, d.n_steps
        self.n_batch = d.n_envs * d.n_steps
        self.n_batch_global = self.n_batch * max(1, d.world_size)
        self.P = self.tensor_size("params_trainable")
        self.Pq = self.tensor_size("params")
        if activation != "tanh":
            self.activation = activation

    def close(self):
        if self._h:
            self.lib.ppo_core_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights
    def load_meta_txt(self, path):
        _check(self.lib, self.lib.ppo_core_load_meta_txt(self._h, path.encode()))

    @property
    def vf_clip(self) -> str:
        """The core's value loss: "shared" (the policy clip range), "none" (no clipping) or "separate" (cliprange_vf)."""
        r = self.lib.ppo_core_vf_clip(self._h)
        if r < 0:
            _check(self.lib, r)
        return VF_CLIP_NAMES[r]

    @vf_clip.setter
    def vf_clip(self, mode: str):
        if mode not in VF_CLIP_MODES:
            raise ValueError(f"vf_clip must be one of {sorted(VF_CLIP_MODES)}, not {mode!r}")
        _check(self.lib, self.lib.ppo_core_set_vf_clip(self._h, VF_CLIP_MODES[mode]))

    @property
    def activation(self) -> str:
        """The core's hidden-layer activation: "tanh" or "relu"."""
        r = self.lib.ppo_core_activation(self._h)
        if r < 0:
            _check(self.lib, r)
        return ACTIVATION_NAMES[r]

    @activation.setter
    def activation(self, act: str):
        if act not in ACTIVATIONS:
            raise ValueError(f"activation must be one of {sorted(ACTIVATIONS)}, not {act!r}")
        _check(self.lib, self.lib.ppo_core_set_activation(self._h, ACTIVATIONS[act]))

    @property
    def action_space(self) -> str:
        """The core's policy head: "box" (Gaussian), "discrete" (categorical over act_dim logits), "multi_discrete" (one categorical
        per slice of the logits) or "multi_binary" (a Bernoulli per logit)."""
        r = self.lib.ppo_core_action_space(self._h)
        if r < 0:
            _check(self.lib, r)
        return ACTION_SPACE_NAMES[r]

    @property
    def nvec(self) -> list:
        """The choices per action column: [act_dim] (discrete), nvec (multi_discrete), 2s (multi_binary); PPOError for a Box core."""
        r = _nvec(self.lib.ppo_core_action_nvec, self._h)
        if isinstance(r, int):
            _check(self.lib, r)
        return r

    @property
    def action_masking(self) -> bool:
        """Invalid-action masks on this core (Discrete / MultiDiscrete only): the *_masked calls and mask= / masks= arguments, and the
        "action_masks" rollout buffer.  Off at creation."""
        r = self.lib.ppo_core_action_masking(self._h)
        if r < 0:
            _check(self.lib, r)
        return bool(r)

    @action_masking.setter
    def action_masking(self, on: bool):
        _check(self.lib, self.lib.ppo_core_set_action_masking(self._h, int(bool(on))))

    def graph_builds(self) -> int:
        """CUDA graphs captured and instantiated since the core was created."""
        n = C.c_uint64()
        _check(self.lib, self.lib.ppo_core_graph_builds(self._h, C.byref(n)))
        return n.value

    def init_orthogonal(self, seed=0):
        _check(self.lib, self.lib.ppo_core_init_orthogonal(self._h, seed))

    def load_checkpoint_data(self, prefix):
        _check(self.lib, self.lib.ppo_core_load_checkpoint_data(self._h, prefix.encode()))

    def save_checkpoint_data(self, prefix):
        _check(self.lib, self.lib.ppo_core_save_checkpoint_data(self._h, prefix.encode()))

    def tensor_size(self, name):
        n = self.lib.ppo_core_tensor_size(self._h, name.encode())
        if n < 0:
            _check(self.lib, n)
        return n

    def get_tensor(self, name):
        out = np.zeros(self.tensor_size(name), np.float32)
        _check(self.lib, self.lib.ppo_core_get_tensor(self._h, name.encode(), out.ctypes.data, out.size))
        return out

    def set_tensor(self, name, value):
        v = _f32(value).ravel()
        _check(self.lib, self.lib.ppo_core_set_tensor(self._h, name.encode(), v.ctypes.data, v.size))

    def sync(self):
        _check(self.lib, self.lib.ppo_core_sync(self._h))

    @property
    def stream(self):
        return self.lib.ppo_core_stream(self._h)

    def counters(self, reset=False):
        c = Counters()
        _check(self.lib, self.lib.ppo_core_counters(self._h, C.byref(c), int(reset)))
        return dict(kernel_launches=c.kernel_launches, graph_launches=c.graph_launches, h2d_bytes=c.h2d_bytes, d2h_bytes=c.d2h_bytes)

    # ---- policy
    def policy_step(self, obs, eps=None, mask=None):
        obs = _f32(obs)
        n = obs.shape[0]
        e = None if eps is None else _f32(eps)
        act, val, nlp = np.zeros((n, self.AW), np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        if mask is None:
            _check(self.lib, self.lib.ppo_policy_step(self._h, _addr(obs), n, _addr(e), _addr(act), _addr(val), _addr(nlp), PPO_HOST))
        else:
            m = _mask(mask, n, self.A)
            _check(self.lib, self.lib.ppo_policy_step_masked(self._h, _addr(obs), n, _addr(e), _addr(m), _addr(act), _addr(val), _addr(nlp), PPO_HOST))
        return act, val, nlp

    def policy_value(self, obs):
        obs = _f32(obs)
        val = np.zeros(obs.shape[0], np.float32)
        _check(self.lib, self.lib.ppo_policy_value(self._h, _addr(obs), obs.shape[0], _addr(val), PPO_HOST))
        return val

    def policy_mean(self, obs, mask=None):
        obs = _f32(obs)
        act = np.zeros((obs.shape[0], self.AW), np.float32)
        if mask is None:
            _check(self.lib, self.lib.ppo_policy_mean(self._h, _addr(obs), obs.shape[0], _addr(act), PPO_HOST))
        else:
            m = _mask(mask, obs.shape[0], self.A)
            _check(self.lib, self.lib.ppo_policy_mean_masked(self._h, _addr(obs), obs.shape[0], _addr(m), _addr(act), PPO_HOST))
        return act

    # ---- VecNormalize
    def vecnorm_reset(self, raw_obs):
        raw = _f32(raw_obs)
        out = np.zeros_like(raw)
        _check(self.lib, self.lib.ppo_vecnorm_reset(self._h, _addr(raw), _addr(out), PPO_HOST))
        return out

    def vecnorm_step(self, raw_obs, raw_rew, done):
        raw, rew, dn = _f32(raw_obs), _f32(raw_rew).ravel(), _f32(done).ravel()
        obs, r = np.zeros_like(raw), np.zeros_like(rew)
        _check(self.lib, self.lib.ppo_vecnorm_step(self._h, _addr(raw), _addr(rew), _addr(dn), _addr(obs), _addr(r), PPO_HOST))
        return obs, r

    def vecnorm_replay(self, raw_obs, raw_rew, done):
        """T consecutive vecnorm_step calls on a recorded trajectory [T, n_envs, O] in four launches."""
        raw = _f32(raw_obs)
        T = raw.shape[0]
        rew, dn = _f32(raw_rew).reshape(T, -1), _f32(done).reshape(T, -1)
        obs, r = np.zeros_like(raw), np.zeros_like(rew)
        _check(self.lib, self.lib.ppo_vecnorm_replay(self._h, _addr(raw), _addr(rew), _addr(dn), T, _addr(obs), _addr(r), PPO_HOST))
        return obs, r

    def vecnorm_stats(self):
        om, ov = np.zeros(self.O, np.float32), np.zeros(self.O, np.float32)
        rm, rv = np.zeros(1, np.float32), np.zeros(1, np.float32)
        oc, rc = C.c_double(), C.c_double()
        _check(self.lib, self.lib.ppo_vecnorm_get_stats(self._h, _addr(om), _addr(ov), C.byref(oc), _addr(rm), _addr(rv), C.byref(rc)))
        return dict(obs_mean=om, obs_var=ov, obs_count=oc.value, ret_mean=rm, ret_var=rv, ret_count=rc.value)

    def vecnorm_set_stats(self, obs_mean, obs_var, obs_count, ret_mean, ret_var, ret_count):
        om, ov, rm, rv = _f32(obs_mean), _f32(obs_var), _f32(ret_mean).ravel(), _f32(ret_var).ravel()
        _check(self.lib, self.lib.ppo_vecnorm_set_stats(self._h, _addr(om), _addr(ov), obs_count, _addr(rm), _addr(rv), ret_count))

    def vecnorm_set_training(self, training):
        _check(self.lib, self.lib.ppo_vecnorm_set_training(self._h, int(training)))

    def running_stats_update(self, mean, var, count, batch):
        m, v, b = _f32(mean).copy(), _f32(var).copy(), _f32(batch)
        cnt = C.c_double(count)
        _check(self.lib, self.lib.ppo_running_stats_update(self._h, _addr(m), _addr(v), C.byref(cnt), b.shape[1], _addr(b), b.shape[0], PPO_HOST))
        return m, v, cnt.value

    def matrix_clamp(self, x, lo, hi):
        x = _f32(x)
        out = np.zeros_like(x)
        _check(self.lib, self.lib.ppo_matrix_clamp(self._h, _addr(x), x.size, lo, hi, _addr(out), PPO_HOST))
        return out

    # ---- GAE
    def gae(self, rewards, values, dones, last_values, last_dones, gamma, lam):
        r, v, d, lv, ld = _f32(rewards), _f32(values), _f32(dones), _f32(last_values), _f32(last_dones)
        if _is_dev(rewards):
            raise TypeError("use gae_device for CUDA tensors")
        T, N = r.shape
        adv, ret = np.zeros((T, N), np.float32), np.zeros((T, N), np.float32)
        _check(self.lib, self.lib.ppo_gae(self._h, _addr(r), _addr(v), _addr(d), _addr(lv), _addr(ld), T, N, gamma, lam, _addr(adv), _addr(ret), PPO_HOST))
        return adv, ret

    def gae_device(self, rewards, values, dones, last_values, last_dones, gamma, lam, advs, returns):
        T, N = rewards.shape
        _check(self.lib, self.lib.ppo_gae(self._h, _addr(rewards), _addr(values), _addr(dones), _addr(last_values), _addr(last_dones),
                                          T, N, gamma, lam, _addr(advs), _addr(returns), PPO_DEVICE))

    # ---- rollout
    def runner_reset(self, raw_obs, mask=None):
        raw = _f32(raw_obs)
        if mask is None:
            _check(self.lib, self.lib.ppo_runner_reset(self._h, _addr(raw), PPO_HOST))
        else:
            m = _mask(mask, self.n_envs, self.A)
            _check(self.lib, self.lib.ppo_runner_reset_masked(self._h, _addr(raw), _addr(m), PPO_HOST))

    def runner_act(self, t, out: Optional[np.ndarray] = None):
        act = out if out is not None else np.zeros((self.n_envs, self.AW), np.float32)
        _check(self.lib, self.lib.ppo_runner_act(self._h, t, _addr(act), PPO_HOST))
        return act

    def runner_observe(self, t, raw_obs, raw_rew, done, mask=None):
        raw, rew, dn = _f32(raw_obs), _f32(raw_rew).ravel(), _f32(done).ravel()
        if mask is None:
            _check(self.lib, self.lib.ppo_runner_observe(self._h, t, _addr(raw), _addr(rew), _addr(dn), PPO_HOST))
        else:
            m = _mask(mask, self.n_envs, self.A)
            _check(self.lib, self.lib.ppo_runner_observe_masked(self._h, t, _addr(raw), _addr(rew), _addr(dn), _addr(m), PPO_HOST))

    def runner_finish(self):
        _check(self.lib, self.lib.ppo_runner_finish(self._h))

    def runner_rollout_replay(self, raw_obs, raw_rew, done, actions_out: Optional[np.ndarray] = None):
        """The act/observe loop of a whole rollout in one C call, the host env being a recorded trajectory."""
        raw, rew, dn = _f32(raw_obs), _f32(raw_rew), _f32(done)
        _check(self.lib, self.lib.ppo_runner_rollout_replay(self._h, _addr(raw), _addr(rew), _addr(dn),
                                                            _addr(actions_out) if actions_out is not None else None))

    def runner_rollout_host(self, step_fn):
        """ppo_runner_rollout_host with a Python env: step_fn(t, actions[n_envs, AW]) -> (raw_obs, raw_rew, done) or None to abort."""
        n = self.n_envs
        keep = {}
        fpp = C.POINTER(C.POINTER(C.c_float))

        @C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_float), fpp, fpp, fpp)
        def cb(_user, t, actions, po, pr, pd):
            act = np.ctypeslib.as_array(actions, (n, self.AW))
            out = step_fn(t, act)
            if out is None:
                return 1
            keep["o"], keep["r"], keep["d"] = (_f32(x).ravel() for x in out)  # alive until the next call
            po[0] = keep["o"].ctypes.data_as(C.POINTER(C.c_float))
            pr[0] = keep["r"].ctypes.data_as(C.POINTER(C.c_float))
            pd[0] = keep["d"].ctypes.data_as(C.POINTER(C.c_float))
            return 0

        actions = np.zeros((n, self.AW), np.float32)
        _check(self.lib, self.lib.ppo_runner_rollout_host(self._h, C.cast(cb, C.c_void_p), None, _addr(actions)))

    def synth_env_reset(self):
        _check(self.lib, self.lib.ppo_synth_env_reset(self._h))

    def rollout_synthetic(self):
        _check(self.lib, self.lib.ppo_rollout_synthetic(self._h))

    def rollout_get(self, name):
        w = self.A if name == "action_masks" else BUFFER_WIDTH[name] or (self.O if name == "obs" else self.AW)
        out = np.zeros((self.n_batch, w), np.float32)
        _check(self.lib, self.lib.ppo_rollout_get(self._h, name.encode(), _addr(out), out.size))
        return out

    def rollout_set(self, name, value):
        v = _f32(value)
        _check(self.lib, self.lib.ppo_rollout_set(self._h, name.encode(), _addr(v), v.size))

    # ---- update
    def shuffle_seed(self, seed):
        _check(self.lib, self.lib.ppo_shuffle_seed(self._h, seed))

    def train_update(self, lr, cliprange, want_losses=True, cliprange_vf=None):
        out = np.zeros(5, np.float32) if want_losses else None
        if cliprange_vf is None:
            _check(self.lib, self.lib.ppo_train_update(self._h, lr, cliprange, _addr(out)))
        else:
            _check(self.lib, self.lib.ppo_train_update_vf(self._h, lr, cliprange, cliprange_vf, _addr(out)))
        return out

    def train_set_permutation(self, perm):
        p = np.ascontiguousarray(perm, np.int32)
        _check(self.lib, self.lib.ppo_train_set_permutation(self._h, p.ctypes.data, p.size))

    def train_get_permutation(self, epoch):
        out = np.zeros(self.n_batch_global, np.int32)
        _check(self.lib, self.lib.ppo_train_get_permutation(self._h, epoch, out.ctypes.data, out.size))
        return out

    def train_minibatch(self, k, lr, cliprange, cliprange_vf=None):
        losses, grads = np.zeros(5, np.float32), np.zeros(self.P, np.float32)
        if cliprange_vf is None:
            _check(self.lib, self.lib.ppo_train_minibatch(self._h, k, lr, cliprange, _addr(losses), _addr(grads)))
        else:
            _check(self.lib, self.lib.ppo_train_minibatch_vf(self._h, k, lr, cliprange, cliprange_vf, _addr(losses), _addr(grads)))
        return losses, grads

    def advnorm(self, returns, values):
        r, v = _f32(returns).ravel(), _f32(values).ravel()
        out = np.zeros_like(r)
        _check(self.lib, self.lib.ppo_advnorm(self._h, _addr(r), _addr(v), r.size, _addr(out)))
        return out

    def loss_grad(self, obs, actions, advs, returns, old_neglogp, old_values, cliprange, cliprange_vf=None, masks=None):
        o, a = _f32(obs), _f32(actions)
        ad, r, on, ov = _f32(advs).ravel(), _f32(returns).ravel(), _f32(old_neglogp).ravel(), _f32(old_values).ravel()
        grads, losses = np.zeros(self.P, np.float32), np.zeros(5, np.float32)
        if masks is not None:
            m = _mask(masks, o.shape[0], self.A)
            _check(self.lib, self.lib.ppo_loss_grad_masked(self._h, _addr(o), _addr(a), _addr(m), _addr(ad), _addr(r), _addr(on), _addr(ov),
                                                           o.shape[0], cliprange, float("nan") if cliprange_vf is None else cliprange_vf,
                                                           _addr(grads), _addr(losses)))
            return grads, losses
        args = (self._h, _addr(o), _addr(a), _addr(ad), _addr(r), _addr(on), _addr(ov), o.shape[0], cliprange)
        if cliprange_vf is None:
            _check(self.lib, self.lib.ppo_loss_grad(*args, _addr(grads), _addr(losses)))
        else:
            _check(self.lib, self.lib.ppo_loss_grad_vf(*args, cliprange_vf, _addr(grads), _addr(losses)))
        return grads, losses

    def learn_update_synthetic(self, lr, cliprange, want_losses=True):
        out = np.zeros(5, np.float32) if want_losses else None
        _check(self.lib, self.lib.ppo_learn_update_synthetic(self._h, lr, cliprange, _addr(out)))
        return out

    def kernel_family(self, which="train"):
        r = self.lib.ppo_core_kernel_family(self._h, which.encode())
        return r.decode() if r else None

    def profile_kernel(self, which, iters=50):
        ms, n = C.c_float(), C.c_int()
        _check(self.lib, self.lib.ppo_profile_kernel(self._h, which.encode(), iters, C.byref(ms), C.byref(n)))
        return ms.value

    # ---- multi-GPU
    def comm_init(self, unique_id: bytes, rank: int, world_size: int):
        _check(self.lib, self.lib.ppo_comm_init(self._h, unique_id, rank, world_size))

    def comm_ipc_handle(self) -> bytes:
        buf = C.create_string_buffer(_lib.PPO_IPC_HANDLE_BYTES)
        _check(self.lib, self.lib.ppo_comm_ipc_handle(self._h, buf))
        return buf.raw

    def comm_ipc_open(self, handles, world_size: int):
        blob = b"".join(handles)
        assert len(blob) == world_size * _lib.PPO_IPC_HANDLE_BYTES
        _check(self.lib, self.lib.ppo_comm_ipc_open(self._h, blob, world_size))

    def comm_set_p2p(self, enable: bool):
        _check(self.lib, self.lib.ppo_comm_set_p2p(self._h, int(enable)))

    def comm_error(self) -> bool:
        return bool(self.lib.ppo_comm_error(self._h))
