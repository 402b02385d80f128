"""Discrete action spaces: the categorical policy head (Stable-Baselines' CategoricalProbabilityDistribution, ppo_action_space).

The reference is an fp64 PyTorch autograd restatement of the PPO2 loss with a categorical head: neglogp from log_softmax,
the entropy exactly as Stable-Baselines writes it (a0 = l - max l, z = sum exp a0, p = exp a0 / z, H = sum p (log z - a0)),
TensorFlow's tie rules for the clipped surrogate and the value loss, Gumbel-max sampling with ties to the first index.
CPU tests: both graph readers on the writer's files and hand edits, the layout and the checkpoint order, the index writer,
the writer's unchanged output without action_space, and the host bandit env.  GPU tests (the F and T families, tanh and
ReLU): policy steps with supplied uniforms and with Philox noise, loss and gradients, whole updates against an fp64 learner,
the host-env protocol, family selection, checkpoints and the CLI (test_multi_gpu_parity.py: sharded discrete updates).  No
real Stable-Baselines Discrete export is available, so the reader rule is checked against the writer's files and hand edits."""
import hashlib
import os
import subprocess
from functools import partial

import numpy as np
import pytest
import torch

from conftest import ROOT, load_weights, rel_err
from ppo_cpp_b200 import meta_graph as mg
from test_abi_cpu import _parse_bundle_index
from test_vf_clip_and_schedules import _tf_clip, _tf_max, learner_ref, value_loss

TOL = 1e-5
ENT = 0.01
O, N = 6, 5  # observation width, number of actions (not a multiple of 4: the Philox blocks have a tail)
FT = [((), "fused"), (("PPO_DISABLE_FUSED",), "tile")]


# ------------------------------------------------------------------ layout and the fp64 reference
def layout(h1, h2, o=O, n=N):
    lay = mg.param_layout(o, n, h1, h2, action_space="discrete")
    order = [t for t in mg.TENSOR_ORDER[:mg.N_TRAINABLE_TENSORS] if t != mg.LOGSTD]
    return [lay[t] for t in order], lay["model/q/w"][0], lay["__total__"][0]


def rand_params(rng, h1, h2, o=O, n=N, head_scale=1.0):
    _, P, Pq = layout(h1, h2, o, n)
    p = (rng.standard_normal(Pq) * min(0.3, 1.5 / np.sqrt(max(h1, h2)))).astype(np.float32)
    lay = mg.param_layout(o, n, h1, h2, action_space="discrete")
    off = lay["model/pi/w"][0]
    p[off:off + h2 * n] *= 4.0 * head_scale  # logits of O(1) spread
    return p


def _act(name):
    return torch.tanh if name == "tanh" else torch.relu


def forward_ref(params, obs, activation, h1, h2, o=O, n=N):
    lay, _, _ = layout(h1, h2, o, n)
    t = [params.astype(np.float64)[off:off + int(np.prod(s))].reshape(s) for off, s in lay]
    f = np.tanh if activation == "tanh" else (lambda z: np.maximum(z, 0.0))
    x = obs.astype(np.float64)
    logits = f(f(x @ t[0] + t[1]) @ t[4] + t[5]) @ t[10] + t[11]
    v = (f(f(x @ t[2] + t[3]) @ t[6] + t[7]) @ t[8] + t[9])[:, 0]
    return logits, v


def neglogp_ref(logits, a):
    mx = logits.max(1, keepdims=True)
    lse = np.log(np.exp(logits - mx).sum(1)) + mx[:, 0]
    return lse - logits[np.arange(len(a)), a]


def loss_grad_ref(params, obs, act, adv, ret, old_nlp, old_v, cr, activation, h1, h2, ent_coef=ENT, vf_coef=0.5, o=O, n=N):
    lay, P, _ = layout(h1, h2, o, n)
    p = torch.tensor(np.asarray(params[:P], np.float64), requires_grad=True)
    pi0w, pi0b, vf0w, vf0b, pi1w, pi1b, vf1w, vf1b, vfw, vfb, piw, pib = [p[off:off + int(np.prod(s))].reshape(s) for off, s in lay]
    f = _act(activation)
    x = torch.tensor(np.asarray(obs, np.float64))
    a = torch.tensor(np.asarray(act).reshape(-1).astype(np.int64))
    adv, R, onl, ov = (torch.tensor(np.asarray(z, np.float64).ravel()) for z in (adv, ret, old_nlp, old_v))
    logits = f(f(x @ pi0w + pi0b) @ pi1w + pi1b) @ piw + pib
    v = (f(f(x @ vf0w + vf0b) @ vf1w + vf1b) @ vfw + vfb)[:, 0]
    nlp = -torch.log_softmax(logits, 1).gather(1, a[:, None])[:, 0]
    ratio = torch.exp(onl - nlp)
    pg = _tf_max(-adv * ratio, -adv * _tf_clip(ratio, torch.tensor(1.0 - cr, dtype=torch.float64),
                                                torch.tensor(1.0 + cr, dtype=torch.float64))).mean()
    vf = 0.5 * value_loss(v, ov, R, "shared", cr, 0.0).mean()
    a0 = logits - logits.max(1, keepdim=True)[0]
    z = torch.exp(a0).sum(1, keepdim=True)
    ent = ((torch.exp(a0) / z) * (torch.log(z) - a0)).sum(1).mean()
    loss = pg - ent * ent_coef + vf * vf_coef
    loss.backward()
    with torch.no_grad():
        kl = 0.5 * ((nlp - onl) ** 2).mean()
        cf = ((ratio - 1.0).abs() > cr).double().mean()
    return p.grad.numpy().copy(), np.array([pg.item(), vf.item(), ent.item(), kl.item(), cf.item()])


def batch(rng, params, activation, h1, h2, B):
    obs = rng.standard_normal((B, O)).astype(np.float32)
    logits, v = forward_ref(params, obs, activation, h1, h2)
    prob = np.exp(logits - logits.max(1, keepdims=True))
    prob /= prob.sum(1, keepdims=True)
    act = np.array([rng.choice(N, p=q) for q in prob])
    old_nlp = (neglogp_ref(logits, act) + 0.1 * rng.standard_normal(B)).astype(np.float32)
    old_v = (v + 0.3 * rng.standard_normal(B)).astype(np.float32)
    ret = (v + 0.3 + 0.5 * rng.standard_normal(B)).astype(np.float32)
    adv = rng.standard_normal(B).astype(np.float32)
    return obs, act.astype(np.float32)[:, None], adv, ret, old_nlp, old_v


def gumbel_fixture(rng, logits):
    """Uniforms u whose Gumbel-perturbed logits l - log(-log u) have a maximum at least 1e-3 above the runner-up (so fp32
    rounding cannot change the index), with u = 0 (never taken) in column 1 of every tenth row."""
    B = logits.shape[0]
    u = rng.uniform(0.0, 1.0, (B, N))
    u[::10, 1] = 0.0
    for _ in range(100):
        with np.errstate(divide="ignore"):
            g = logits - np.log(-np.log(u))
        s = np.sort(g, 1)
        bad = s[:, -1] - s[:, -2] < 1e-3
        if not bad.any():
            break
        u[bad] = rng.uniform(0.0, 1.0, (int(bad.sum()), N))
    return u.astype(np.float32), np.argmax(g, 1)


# ------------------------------------------------------------------ CPU: the graph readers and the writer
def _tensors(h1=4, h2=5, o=O, n=N):
    rng = np.random.default_rng(1)
    return {name: rng.standard_normal(s).astype(np.float32) for name, (off, s) in mg.param_layout(o, n, h1, h2).items() if name != "__total__"}


def _graph(tmp_path, action_space, name=None, activation=None):
    path = str(tmp_path / (name or f"g_{action_space}.meta.txt"))
    mg.write_meta_txt(path, _tensors(), ent_coef=ENT, action_space=action_space, activation=activation)
    return path


def test_writer_without_action_space_is_unchanged(tmp_path):
    """Without action_space the writer's output is byte for byte what it was before (the digest test_activation pins)."""
    tensors, _ = load_weights("graph_4_5_init.npz")
    path = str(tmp_path / "u.meta.txt")
    mg.write_meta_txt(path, tensors, ent_coef=0.0007160293171182275)
    assert hashlib.sha256(open(path, "rb").read()).hexdigest() == "8ef88a589ddf33dea18f33440cfdbceab404d08437f76c386d84045f04457d9f"


@pytest.mark.parametrize("space,dtype", [(None, None), ("box", None), ("discrete", "DT_INT64"), ("discrete", "DT_INT32")])
def test_readers_classify_the_action_space(tmp_path, space, dtype):
    from ppo_cpp_b200 import core
    path = _graph(tmp_path, space, activation="relu")
    text = open(path, encoding="latin-1").read()
    assert ("loss/action_ph" in text) == (space is not None) and (mg.LOGSTD in text) == (space != "discrete")
    if dtype == "DT_INT32":
        with open(path, "w", encoding="latin-1") as f:
            f.write(text.replace("type: DT_INT64", "type: DT_INT32"))
    want = space or "box"
    assert mg.parse_meta_txt(path).action_space == mg.meta_action_space(path) == core.meta_action_space(path) == want
    assert core.meta_activation(path) == "relu"
    info, params = core.meta_parse(path)
    lay = mg.param_layout(O, N, 4, 5, action_space=want)
    assert (info.obs_dim, info.act_dim, info.hidden1, info.hidden2) == (O, N, 4, 5)
    assert info.n_params_total == lay["__total__"][0] and info.n_params_trainable == lay["model/q/w"][0]
    np.testing.assert_array_equal(params, mg.parse_meta_txt(path).flat_params())


EDITS = {  # hand edits the readers must refuse
    "logstd_with_int_placeholder": ("box", "type: DT_FLOAT\n      }\n    }\n    attr {\n      key: \"shape\"\n      value {\n        shape {\n          dim {\n            size: -1",
                                    "type: DT_INT64\n      }\n    }\n    attr {\n      key: \"shape\"\n      value {\n        shape {\n          dim {\n            size: -1"),
    "no_logstd_with_float_placeholder": ("discrete", "type: DT_INT64", "type: DT_FLOAT"),
    "discrete_rank_2": ("discrete", "            size: -1\n          }\n", "            size: -1\n          }\n          dim {\n            size: 5\n          }\n"),
}


@pytest.mark.parametrize("edit", sorted(EDITS))
def test_readers_reject_a_contradicting_placeholder(tmp_path, edit):
    from ppo_cpp_b200 import core
    space, old, new = EDITS[edit]
    path = _graph(tmp_path, space)
    text = open(path, encoding="latin-1").read()
    assert text.count(old) == 1
    with open(path, "w", encoding="latin-1") as f:
        f.write(text.replace(old, new))
    with pytest.raises(ValueError, match="loss/action_ph"):
        mg.parse_meta_txt(path)
    for fn in (core.meta_action_space, core.meta_parse):
        with pytest.raises(core.PPOError, match=r"\[-4\].*loss/action_ph"):
            fn(path)


def test_param_layout_and_checkpoint_order(tmp_path):
    box, disc = mg.param_layout(O, N, 8, 8), mg.param_layout(O, N, 8, 8, action_space="discrete")
    assert mg.LOGSTD not in disc and len(disc) == 15  # 14 tensors + __total__
    assert disc["__total__"][0] == box["__total__"][0] - N
    for t in mg.TENSOR_ORDER:  # graph gradient order kept; everything behind logstd moves down by its size
        if t != mg.LOGSTD:
            assert disc[t][1] == box[t][1] and disc[t][0] == box[t][0] - (N if box[t][0] > box[mg.LOGSTD][0] else 0)
    shapes = {t: s for t, (o, s) in disc.items() if t != "__total__"}
    payload = {t: np.random.default_rng(2).standard_normal(s).astype(np.float32) for t, s in shapes.items()}
    raw = np.concatenate([payload[t].ravel() for t in mg.CKPT_ORDER if t in payload])
    raw.tofile(tmp_path / "c.data-00000-of-00001")
    got = mg.read_checkpoint_data(str(tmp_path / "c.data-00000-of-00001"), shapes)
    assert list(got) == [t for t in mg.CKPT_ORDER if t != mg.LOGSTD]
    for t in shapes:
        np.testing.assert_array_equal(got[t], payload[t])
    with pytest.raises(ValueError):
        mg.param_layout(O, N, 8, 8, action_space="multidiscrete")


def test_index_writer_discrete_round_trip(tmp_path):
    import ctypes as C
    from ppo_cpp_b200 import _lib
    lib = _lib.load()
    disc = mg.param_layout(O, N, 64, 64, action_space="discrete")
    n = disc["__total__"][0]
    data = np.arange(n, dtype=np.float32)
    fp = data.ctypes.data_as(C.POINTER(C.c_float))
    assert lib.ppo_checkpoint_write_index_ex(str(tmp_path / "d").encode(), _lib.PPO_ACTION_DISCRETE, O, N, 64, 64, fp, n) == 0
    ent = _parse_bundle_index(open(tmp_path / "d.index", "rb").read())
    names = [t for t in mg.CKPT_ORDER if t != mg.LOGSTD]
    assert list(ent)[1:] == names
    off = 0
    for t in names:
        assert tuple(ent[t]["shape"]) == disc[t][1] and ent[t].get("offset", 0) == off and ent[t]["size"] == 4 * int(np.prod(disc[t][1]))
        off += ent[t]["size"]
    assert off == 4 * n
    # the Box form of the _ex writer is the old writer, byte for byte
    m = mg.param_layout(O, N, 64, 64)["__total__"][0]
    full = np.arange(m, dtype=np.float32)
    ff = full.ctypes.data_as(C.POINTER(C.c_float))
    assert lib.ppo_checkpoint_write_index_ex(str(tmp_path / "b").encode(), _lib.PPO_ACTION_BOX, O, N, 64, 64, ff, m) == 0
    assert lib.ppo_checkpoint_write_index(str(tmp_path / "a").encode(), O, N, 64, 64, ff, m) == 0
    assert open(tmp_path / "a.index", "rb").read() == open(tmp_path / "b.index", "rb").read()
    assert lib.ppo_checkpoint_write_index_ex(str(tmp_path / "e").encode(), _lib.PPO_ACTION_DISCRETE, O, N, 64, 64, ff, m) == -1  # 15-tensor payload
    assert lib.ppo_checkpoint_write_index_ex(str(tmp_path / "f").encode(), 2, O, N, 64, 64, fp, n) == -1


def test_host_bandit_env(tmp_path):
    """The CLI's Discrete(4) env: one-hot contexts, reward 1 exactly for the action (c + 1) mod n, 16-step episodes, and
    PPO2's action width of 1 for a discrete env (env.hpp action_width)."""
    src = tmp_path / "b.cpp"
    src.write_text('#include "env_bandit.hpp"\n#include <cstdio>\nint main() {\n  BanditEnv e(7, 0, 4);\n  Mat obs = e.reset();\n'
                   '  int ok = e.get_action_space() == Env::SPACE_DISCRETE() && e.get_action_space_size() == 4 && action_width(e) == 1;\n'
                   '  float good = 0, bad = 0, dones = 0;\n  for (int t = 0; t < 64; ++t) {\n    int c = 0;\n'
                   '    for (int k = 0; k < 4; ++k) { ok &= obs(0, k) == (obs(0, k) > 0.5f ? 1.f : 0.f); if (obs(0, k) > 0.5f) c = k; }\n'
                   '    Mat a(1, 1); a(0, 0) = (float)((c + 1 + (t & 1)) % 4);\n    auto r = e.step(a);\n'
                   '    (t & 1 ? bad : good) += r[1](0, 0); dones += r[2](0, 0); obs = r[0];\n  }\n'
                   '  std::printf("%d %g %g %g\\n", ok, good, bad, dones);\n  return 0;\n}\n')
    exe = tmp_path / "b"
    subprocess.run(["g++", "-std=c++14", "-O1", "-I", os.path.join(ROOT, "ppo_cpp_b200", "host"), "-o", str(exe), str(src)], check=True)
    ok, good, bad, dones = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert (int(ok), float(good), float(bad), float(dones)) == (1, 32.0, 0.0, 4.0)


# ------------------------------------------------------------------ GPU
def _core(core_mod, monkeypatch, env=(), **kw):
    for e in env:
        monkeypatch.setenv(e, "1")
    kw.setdefault("obs_dim", O)
    kw.setdefault("act_dim", N)
    c = core_mod.PPOCore(action_space="discrete", **kw)
    for e in env:
        monkeypatch.delenv(e)
    assert c.action_space == "discrete"
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ["tanh", "relu"])
@pytest.mark.parametrize("env,fam", FT)
def test_policy_step_with_given_uniforms_vs_fp64(monkeypatch, env, fam, activation):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(3)
    B = 3000
    p = rand_params(rng, 64, 64)
    obs = rng.standard_normal((B, O)).astype(np.float32)
    logits, v64 = forward_ref(p, obs, activation, 64, 64)
    u, want = gumbel_fixture(rng, logits)
    c = _core(core_mod, monkeypatch, env, activation=activation, hidden1=64, hidden2=64, n_envs=B, n_steps=2, nminibatches=1)
    assert fam in c.kernel_family("policy") and fam in c.kernel_family("train"), c.kernel_family("policy")
    c.set_tensor("params", p)
    a, v, nlp = c.policy_step(obs, u)
    assert a.shape == (B, 1) and np.array_equal(a[:, 0], want.astype(np.float32))
    assert not np.any(a[::10, 0] == 1.0)  # u = 0 is never taken
    assert rel_err(nlp, neglogp_ref(logits, want)) < TOL and rel_err(v, v64) < TOL
    s = np.sort(logits, 1)
    sep = s[:, -1] - s[:, -2] > 1e-4
    det = c.policy_mean(obs)
    assert det.shape == (B, 1) and np.array_equal(det[sep, 0], np.argmax(logits, 1)[sep].astype(np.float32))
    # exact ties: equal logits and equal uniforms -> the first index, as TF's ArgMax
    q = p.copy()
    lay = mg.param_layout(O, N, 64, 64, action_space="discrete")
    q[lay["model/pi/w"][0]:lay["model/pi/w"][0] + 64 * N] = 0.0
    q[lay["model/pi/b"][0]:lay["model/pi/b"][0] + N] = 0.25
    c.set_tensor("params", q)
    a, _, nlp = c.policy_step(obs[:64], np.full((64, N), 0.5, np.float32))
    assert np.all(a == 0.0) and np.all(c.policy_mean(obs[:64]) == 0.0)
    assert np.allclose(nlp, np.log(N), rtol=1e-6)
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env,fam", FT)
def test_philox_action_frequencies_match_softmax(monkeypatch, env, fam):
    """Every env sees the same observation: the index frequencies over 200 000 draws match softmax(l) (chi-square at a fixed seed)."""
    from scipy import stats
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(4)
    B = 50000
    p = rand_params(rng, 64, 64, head_scale=0.3)
    obs = np.repeat(rng.standard_normal((1, O)).astype(np.float32), B, 0)
    logits, _ = forward_ref(p, obs[:1], "tanh", 64, 64)
    prob = np.exp(logits[0] - logits[0].max())
    prob /= prob.sum()
    assert prob.min() > 0.02
    c = _core(core_mod, monkeypatch, env, hidden1=64, hidden2=64, n_envs=B, n_steps=2, nminibatches=1, seed=123)
    c.set_tensor("params", p)
    counts = np.zeros(N)
    draws = []
    for _ in range(4):
        a, _, nlp = c.policy_step(obs)
        draws.append(a[:, 0].copy())
        counts += np.bincount(a[:, 0].astype(int), minlength=N)
        assert rel_err(nlp, neglogp_ref(np.repeat(logits, B, 0), a[:, 0].astype(int))) < TOL
    c.close()
    assert not np.array_equal(draws[0], draws[1])  # the step counter advances the stream
    chi2, pval = stats.chisquare(counts, counts.sum() * prob)
    assert pval > 1e-3, (counts / counts.sum(), prob, pval)


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ["tanh", "relu"])
def test_loss_grad_vs_fp64_and_f_equals_t(monkeypatch, activation):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(5)
    h = 64
    p = rand_params(rng, h, h)
    data = batch(rng, p, activation, h, h, 1000)
    g64, l64 = loss_grad_ref(p, *data, 0.2, activation, h, h)
    lay, _, _ = layout(h, h)
    outs = []
    for env, fam in FT:
        c = _core(core_mod, monkeypatch, env, activation=activation, hidden1=h, hidden2=h, n_envs=4, n_steps=8, nminibatches=4, ent_coef=ENT)
        assert fam in c.kernel_family("train")
        assert c.tensor_size("params_trainable") == lay[-1][0] + N
        c.set_tensor("params", p)
        g, l = c.loss_grad(*data, 0.2)
        c.close()
        for t, (off, s) in enumerate(lay):
            sl = slice(off, off + int(np.prod(s)))
            assert rel_err(g[sl], g64[sl]) < TOL, (fam, t, rel_err(g[sl], g64[sl]))
        assert np.allclose(l, l64, rtol=TOL, atol=1e-7), (fam, l, l64)
        outs.append((g, l))
    assert rel_err(outs[0][0], outs[1][0]) < 2e-6 and np.allclose(outs[0][1], outs[1][1], rtol=2e-6, atol=1e-8)
    # the entropy term matters: without it the logits' gradient differs
    g0, _ = loss_grad_ref(p, *data, 0.2, activation, h, h, ent_coef=0.0)
    assert rel_err(g0, g64) > 1e-3


def _replay_rollout(rng, n_envs, n_steps):
    raw = rng.standard_normal((n_steps, n_envs, O)).astype(np.float32)
    rew = rng.standard_normal((n_steps, n_envs)).astype(np.float32)
    done = (rng.uniform(size=(n_steps, n_envs)) < 0.05).astype(np.float32)
    return raw, rew, done


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ["tanh", "relu"])
@pytest.mark.parametrize("env,fam", FT)
@pytest.mark.parametrize("switch", [(), ("PPO_DISABLE_GRAPH",), ("PPO_DISABLE_GPU_SHUFFLE",)])
def test_train_update_vs_fp64_learner(monkeypatch, env, fam, activation, switch):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(21)
    h, n_envs, n_steps, nmb, epochs = 64, 128, 16, 4, 2
    flat = rand_params(rng, h, h)
    raw, rew, done = _replay_rollout(rng, n_envs, n_steps)
    c = _core(core_mod, monkeypatch, env + switch, activation=activation, hidden1=h, hidden2=h, n_envs=n_envs, n_steps=n_steps,
              nminibatches=nmb, noptepochs=epochs, ent_coef=ENT, seed=9)
    assert fam in c.kernel_family("train")
    c.set_tensor("params", flat)
    c.runner_reset(rng.standard_normal((n_envs, O)).astype(np.float32))
    c.runner_rollout_replay(raw, rew, done)
    bufs = {n: c.rollout_get(n) for n in ("obs", "actions", "returns", "values", "neglogpacs")}
    assert bufs["actions"].shape == (n_envs * n_steps, 1)
    c.shuffle_seed(42)
    losses = c.train_update(3.9e-4, 0.2)
    perms = [c.train_get_permutation(e) for e in range(epochs)]
    got = c.get_tensor("params")
    c.close()
    p64, want = learner_ref(flat, bufs, perms, nmb, 3.9e-4, 0.2, partial(loss_grad_ref, activation=activation, h1=h, h2=h))
    _, P, _ = layout(h, h)
    moved = np.abs(p64[:P] - flat[:P]).max()
    assert np.abs(got[:P] - p64[:P]).max() < max(5e-4, 4e-5 * epochs * nmb) * moved
    assert np.abs(got[:P] - p64[:P]).max() < 1e-6 * max(1.0, np.abs(p64[:P]).max()) * epochs * nmb
    assert np.allclose(losses, want, rtol=2e-5, atol=1e-6), (losses, want)


@pytest.mark.gpu
@pytest.mark.parametrize("env,fam", FT)
def test_host_env_protocol_and_replay(monkeypatch, env, fam):
    """ppo_runner_rollout_replay, ppo_runner_rollout_host and the per-call act/observe loop store the same integer actions,
    and those are the per-call policy steps."""
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(8)
    n_envs, n_steps = 96, 12
    flat = rand_params(rng, 64, 64)
    obs0 = rng.standard_normal((n_envs, O)).astype(np.float32)
    raw, rew, done = _replay_rollout(rng, n_envs, n_steps)
    res = []
    for mode in ("replay", "host", "stepwise"):
        c = _core(core_mod, monkeypatch, env, hidden1=64, hidden2=64, n_envs=n_envs, n_steps=n_steps, nminibatches=4, seed=31)
        assert c.kernel_family("rollout") == "per-step kernels"
        c.set_tensor("params", flat)
        c.runner_reset(obs0)
        acts = np.zeros((n_steps, n_envs, 1), np.float32)
        if mode == "replay":
            c.runner_rollout_replay(raw, rew, done, acts)
        elif mode == "host":
            def step(t, a):
                acts[t] = a
                return raw[t], rew[t], done[t]
            c.runner_rollout_host(step)
        else:
            for t in range(n_steps):
                c.runner_act(t, acts[t])
                c.runner_observe(t, raw[t], rew[t], done[t])
            c.runner_finish()
        res.append((acts, {n: c.rollout_get(n) for n in ("obs", "actions", "values", "neglogpacs", "returns")}))
        c.close()
    acts = res[0][0]
    assert np.array_equal(acts, np.round(acts)) and acts.min() >= 0 and acts.max() <= N - 1 and len(np.unique(acts)) == N
    for a, bufs in res:
        assert np.array_equal(a, acts)
        assert np.array_equal(bufs["actions"].reshape(n_envs, n_steps), acts[:, :, 0].T)  # flat layout row = env * n_steps + t
        for k in bufs:
            assert np.array_equal(bufs[k], res[0][1][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("h1,h2", [(4, 5), (64, 64), (256, 256)])
def test_family_selection_and_unsupported_paths(h1, h2):
    from ppo_cpp_b200 import core as core_mod
    kw = dict(obs_dim=18, act_dim=18, hidden1=h1, hidden2=h2, n_envs=1024, n_steps=16, nminibatches=4)
    c = core_mod.PPOCore(action_space="discrete", **kw)
    fams = [c.kernel_family(w) for w in ("train", "policy", "rollout")]
    assert ("train_fused_kernel" in fams[0]) or ("train_tile_kernel" in fams[0]), fams
    assert ("policy_fused_kernel" in fams[1]) or ("policy_tile_kernel" in fams[1]), fams
    assert fams[2] == "per-step kernels"
    for fn in (c.synth_env_reset, c.rollout_synthetic, lambda: c.learn_update_synthetic(3e-4, 0.2)):
        with pytest.raises(core_mod.PPOError, match=r"\[-4\]"):
            fn()
    for name in (mg.LOGSTD, mg.LOGSTD + "/Adam", mg.LOGSTD + "/Adam_1"):
        with pytest.raises(core_mod.PPOError, match=r"\[-1\]"):
            c.tensor_size(name)
    B = 16
    obs = np.zeros((B, 18), np.float32)
    args = (np.zeros(B), np.zeros(B), np.zeros(B), np.zeros(B), 0.2)
    for bad in (18.0, -1.0, 0.5):
        with pytest.raises(core_mod.PPOError, match=r"\[-1\]"):
            c.loss_grad(obs, np.full((B, 1), bad, np.float32), *args)
        with pytest.raises(core_mod.PPOError, match=r"\[-1\]"):
            c.rollout_set("actions", np.full((c.n_batch, 1), bad, np.float32))
    c.close()
    box = core_mod.PPOCore(**kw)
    assert box.action_space == "box"
    box.close()
    with pytest.raises(ValueError):
        core_mod.PPOCore(action_space="multidiscrete")


@pytest.mark.gpu
def test_checkpoint_and_graph_round_trip(tmp_path):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(12)
    kw = dict(obs_dim=O, act_dim=N, hidden1=64, hidden2=64, n_envs=8, n_steps=8, nminibatches=2)
    c = core_mod.PPOCore(action_space="discrete", **kw)
    c.init_orthogonal(3)
    lay = mg.param_layout(O, N, 64, 64, action_space="discrete")
    p0 = c.get_tensor("params")
    assert p0.size == lay["__total__"][0]
    w = p0[lay["model/pi/w"][0]:lay["model/pi/w"][0] + 64 * N].reshape(64, N).astype(np.float64)
    assert np.allclose(w.T @ w, 1e-4 * np.eye(N), atol=1e-8)  # orthogonal at scale 0.01
    p = rand_params(rng, 64, 64)
    c.set_tensor("params", p)
    prefix = str(tmp_path / "ck")
    c.save_checkpoint_data(prefix)
    assert os.path.getsize(prefix + ".data-00000-of-00001") == 4 * p.size
    ent = _parse_bundle_index(open(prefix + ".index", "rb").read())
    assert list(ent)[1:] == [t for t in mg.CKPT_ORDER if t != mg.LOGSTD]
    shapes = {t: s for t, (o, s) in lay.items() if t != "__total__"}
    data = mg.read_checkpoint_data(prefix + ".data-00000-of-00001", shapes)
    for t, (o, s) in lay.items():
        if t != "__total__":
            np.testing.assert_array_equal(data[t], p[o:o + int(np.prod(s))].reshape(s))
    d = core_mod.PPOCore(action_space="discrete", **kw)
    d.load_checkpoint_data(prefix)
    assert np.array_equal(d.get_tensor("params"), p)
    d.close()
    # graphs: the core takes a graph of its own action space only
    g = str(tmp_path / "g64.meta.txt")
    t = {k: rng.standard_normal(s).astype(np.float32) for k, (o, s) in mg.param_layout(O, N, 64, 64).items() if k != "__total__"}
    mg.write_meta_txt(g, t, ent_coef=ENT, action_space="discrete")
    c.load_meta_txt(g)
    assert np.array_equal(c.get_tensor("params"), mg.parse_meta_txt(g).flat_params())
    box = core_mod.PPOCore(**kw)
    with pytest.raises(core_mod.PPOError, match=r"\[-1\].*action space"):
        box.load_meta_txt(g)
    gb = str(tmp_path / "gb.meta.txt")
    mg.write_meta_txt(gb, t, ent_coef=ENT, action_space="box")
    with pytest.raises(core_mod.PPOError, match=r"\[-1\].*action space"):
        c.load_meta_txt(gb)
    box.close()
    c.close()


@pytest.mark.gpu
def test_cli_bandit_train_save_load_eval(tmp_path):
    host = os.path.join(ROOT, "ppo_cpp_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    exe = os.path.join(host, "bin", "ppo_cpp")
    common = ["--env", "bandit", "--threads", "4", "--seed", "5"]
    r = subprocess.run([exe, "-d", str(tmp_path / "exp"), "--id", "d0", "--hidden", "64,64", "--steps", "65536", "--lr", "3e-3",
                        "--num_epochs", "4", "--batch_steps", "512", "--saves", "1", *common], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    ck = tmp_path / "exp" / "checkpoints" / "d0"
    side = [f for f in os.listdir(ck) if f.endswith(".json")]
    assert side and all('"discrete"' in open(ck / f).read() for f in side), side
    prefix = str(ck / side[0][:-len(".json")])
    assert os.path.getsize(prefix + ".data-00000-of-00001") == 4 * mg.param_layout(4, 4, 64, 64, action_space="discrete")["__total__"][0]
    r = subprocess.run([exe, "-p", prefix, "--duration", "0.3", *common], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "episode_reward" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    # a discrete checkpoint on a continuous env is refused
    r = subprocess.run([exe, "-p", prefix, "--duration", "0.3", "--env", "synthetic", "--seed", "5"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0
