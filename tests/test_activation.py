"""The hidden-layer activation read from the graph file (Stable-Baselines' act_fun: tf.tanh or tf.nn.relu, ppo_activation).

The reference is an fp64 PyTorch autograd restatement of the PPO2 loss with torch.relu, whose gradient also masks on
output > 0, as TensorFlow's ReluGrad does.  CPU tests: both graph readers on the writer's files and hand-edited variants, the
writer's unchanged output without activation, and the reference's tie fixture (pre-activations exactly 0).  GPU tests: every
forward path, the persistent rollout, every train family's loss and gradients, whole updates, family selection, switching
the activation of a live core and the host C++ CLI.  (A two-GPU ReLU update is not covered here; no real Stable-Baselines ReLU
export is available, so the reader rule is checked against the writer's files and hand edits of them only.)"""
import hashlib
import os
import subprocess

import numpy as np
import pytest
import torch

import oracle_lib as ol
from conftest import ROOT, load_weights, rel_err
from ppo_cpp_b200 import meta_graph as mg
from test_vf_clip_and_schedules import (HALF_LOG_2PI, HALF_LOG_2PIE, _layout, _tf_clip, _tf_max, rand_params,
                                        tensor_slices, value_loss)

TOL = 1e-5
ENT = 0.0007160293171182275


# ------------------------------------------------------------------ fp64 reference (PyTorch autograd)
def _act(name, mask):
    if name == "tanh":
        return torch.tanh
    if mask == "gt":
        return torch.relu  # d relu / dx = (relu(x) > 0), TensorFlow's ReluGrad
    return lambda z: torch.where(z >= 0, z, torch.zeros_like(z))  # gradient on x >= 0 (a unit at exactly 0 passes it)


def loss_grad_ref(params, obs, act, adv, ret, old_nlp, old_v, cr, activation, h1, h2, ent_coef=ENT, vf_coef=0.5, mask="gt"):
    lay, P = _layout(h1, h2)
    p = torch.tensor(np.asarray(params[:P], np.float64), requires_grad=True)
    T = [p[o:o + int(np.prod(s))].reshape(s) for o, s in lay]
    pi0w, pi0b, vf0w, vf0b, pi1w, pi1b, vf1w, vf1b, vfw, vfb, piw, pib, logstd = T
    f = _act(activation, mask)
    x = torch.tensor(np.asarray(obs, np.float64))
    a = torch.tensor(np.asarray(act, np.float64))
    adv, R, onl, ov = (torch.tensor(np.asarray(z, np.float64).ravel()) for z in (adv, ret, old_nlp, old_v))
    mu = f(f(x @ pi0w + pi0b) @ pi1w + pi1b) @ piw + pib
    v = (f(f(x @ vf0w + vf0b) @ vf1w + vf1b) @ vfw + vfb)[:, 0]
    ls = logstd.reshape(-1)
    nlp = 0.5 * (((a - mu) / torch.exp(ls)) ** 2).sum(1) + HALF_LOG_2PI * a.shape[1] + ls.sum()
    ratio = torch.exp(onl - nlp)
    pg = _tf_max(-adv * ratio, -adv * _tf_clip(ratio, torch.tensor(1.0 - cr, dtype=torch.float64),
                                                torch.tensor(1.0 + cr, dtype=torch.float64))).mean()
    vf = 0.5 * value_loss(v, ov, R, "shared", cr, 0.0).mean()
    ent = (ls + HALF_LOG_2PIE).sum()
    loss = pg - ent * ent_coef + vf * vf_coef
    loss.backward()
    with torch.no_grad():
        kl = 0.5 * ((nlp - onl) ** 2).mean()
        cf = ((ratio - 1.0).abs() > cr).double().mean()
    return p.grad.numpy().copy(), np.array([pg.item(), vf.item(), ent.item(), kl.item(), cf.item()])


def forward_ref(params, obs, activation, h1, h2):
    lay, _ = _layout(h1, h2)
    t = [params.astype(np.float64)[o:o + int(np.prod(s))].reshape(s) for o, s in lay]
    f = np.tanh if activation == "tanh" else (lambda z: np.maximum(z, 0.0))
    x = obs.astype(np.float64)
    mu = f(f(x @ t[0] + t[1]) @ t[4] + t[5]) @ t[10] + t[11]
    v = (f(f(x @ t[2] + t[3]) @ t[6] + t[7]) @ t[8] + t[9])[:, 0]
    return mu, v


def batch(rng, params, activation, h1, h2, B):
    obs = rng.standard_normal((B, 18)).astype(np.float32)
    mu, v = forward_ref(params, obs, activation, h1, h2)
    lay, _ = _layout(h1, h2)
    std = np.exp(params[lay[12][0]:lay[12][0] + 18].astype(np.float64))
    act = (mu + std * rng.standard_normal((B, 18))).astype(np.float32)
    z = (act - mu) / std
    old_nlp = (0.5 * (z * z).sum(1) + 18 * HALF_LOG_2PI + np.log(std).sum() + 0.1 * rng.standard_normal(B)).astype(np.float32)
    old_v = (v + 0.3 * rng.standard_normal(B)).astype(np.float32)
    ret = (v + 0.3 + 0.5 * rng.standard_normal(B)).astype(np.float32)
    adv = rng.standard_normal(B).astype(np.float32)
    return obs, act, adv, ret, old_nlp, old_v


def tie_params(rng, h1, h2):
    """Every fourth hidden unit of each layer has zero bias and a zero weight column: its pre-activation is exactly 0 for
    every input, so relu'(0) decides its gradient (0 under TensorFlow's rule)."""
    p = rand_params(rng, h1, h2)
    lay = mg.param_layout(18, 18, h1, h2)
    for w, b, n_in, n in (("pi_fc0", "pi_fc0", 18, h1), ("vf_fc0", "vf_fc0", 18, h1), ("pi_fc1", "pi_fc1", h1, h2), ("vf_fc1", "vf_fc1", h1, h2)):
        W = p[lay[f"model/{w}/w"][0]:lay[f"model/{w}/w"][0] + n_in * n].reshape(n_in, n)
        W[:, ::4] = 0.0
        p[lay[f"model/{b}/b"][0]:lay[f"model/{b}/b"][0] + n][::4] = 0.0
    return p


def range_params(rng, h):
    """Activations from ~1e-4 to more than 1000 (the U and W families store them as fp16 pieces at their own scale)."""
    p = rand_params(rng, h, h)
    lay = mg.param_layout(18, 18, h, h)
    for t in ("pi_fc0", "vf_fc0"):
        o = lay[f"model/{t}/w"][0]
        W = p[o:o + 18 * h].reshape(18, h)
        W *= np.logspace(-4, 2.2, h)[None, :].astype(np.float32)
    for t in ("pi_fc1", "vf_fc1"):
        o = lay[f"model/{t}/w"][0]
        W = p[o:o + h * h].reshape(h, h)
        W *= np.logspace(-3, 1.6, h)[None, :].astype(np.float32)
    for t in ("pi", "vf"):  # keep the heads O(1)
        o = lay[f"model/{t}/w"][0]
        n = h * (18 if t == "pi" else 1)
        p[o:o + n] *= 1e-3
    return p


# ------------------------------------------------------------------ CPU: the reference and its tie fixture
def test_reference_tie_fixture_separates_gt_from_ge():
    rng = np.random.default_rng(3)
    p = tie_params(rng, 4, 5)
    obs, act, adv, ret, old_nlp, old_v = batch(rng, p, "relu", 4, 5, 64)
    x = obs.astype(np.float64)
    lay, _ = _layout(4, 5)
    W0 = p[lay[0][0]:lay[0][0] + 72].reshape(18, 4).astype(np.float64)
    assert np.all((x @ W0 + p[lay[1][0]:lay[1][0] + 4])[:, 0] == 0.0)  # unit 0: pre-activation exactly 0
    g_gt, l_gt = loss_grad_ref(p, obs, act, adv, ret, old_nlp, old_v, 0.2, "relu", 4, 5, mask="gt")
    g_ge, l_ge = loss_grad_ref(p, obs, act, adv, ret, old_nlp, old_v, 0.2, "relu", 4, 5, mask="ge")
    assert np.array_equal(l_gt, l_ge)  # same forward pass
    sl = tensor_slices(4, 5)
    assert np.all(g_gt[sl[1]][::4] == 0.0) and np.any(g_ge[sl[1]][::4] != 0.0)  # the tied units' bias gradient
    assert rel_err(g_ge, g_gt) > 1e-3


# ------------------------------------------------------------------ CPU: the graph readers
def _graph(tmp_path, activation, name=None, vf_clip=None):
    tensors, _ = load_weights("graph_4_5_init.npz")
    path = str(tmp_path / (name or f"g_{activation}.meta.txt"))
    mg.write_meta_txt(path, tensors, ent_coef=ENT, vf_clip=vf_clip, activation=activation)
    return path


def test_writer_without_activation_is_unchanged(tmp_path):
    """Without activation the writer's output is byte for byte what it was before the forward nodes existed."""
    want = {None: "8ef88a589ddf33dea18f33440cfdbceab404d08437f76c386d84045f04457d9f",
            "separate": "f2e1a04c3e8cf7a6acda86b22e066bb8656170a7d29e49d25172d1e9a9b15560"}
    for vf, digest in want.items():
        path = _graph(tmp_path, None, name=f"u_{vf}.meta.txt", vf_clip=vf)
        assert hashlib.sha256(open(path, "rb").read()).hexdigest() == digest


@pytest.mark.parametrize("activation", [None, "tanh", "relu"])
def test_readers_classify_the_activation(tmp_path, activation):
    from ppo_cpp_b200 import core
    path = _graph(tmp_path, activation, vf_clip="separate")
    want = activation or "tanh"  # no forward nodes: the shipped graph's form
    assert mg.parse_meta_txt(path).activation == want
    assert mg.meta_activation(path) == want
    assert core.meta_activation(path) == want
    assert mg.parse_meta_txt(path).vf_clip == core.meta_vf_clip(path) == "separate"
    info, _ = core.meta_parse(path)
    assert (info.hidden1, info.hidden2) == (4, 5)


def _grad_matmuls(activation):
    """The MatMuls TensorFlow's _MatMulGrad adds to the gradient sub-graph of train_model's hidden layers and heads, as
    in a real PPO2 export: the input gradient dY * W^T (transpose_b, second operand the weight's read) and the weight
    gradient X^T * dY (transpose_a, first operand the layer's input activation)."""
    kind = {"tanh": "Tanh", "relu": "Relu"}[activation]
    acts = {"pi_fc1": f"train_model/{kind}", "pi": f"train_model/{kind}_2", "vf_fc1": f"train_model/{kind}_1", "vf": f"train_model/{kind}_3"}

    def node(name, x, y, flag):
        return (f'  node {{\n    name: "{name}"\n    op: "MatMul"\n    input: "{x}"\n    input: "{y}"\n'
                f'    attr {{\n      key: "T"\n      value {{\n        type: DT_FLOAT\n      }}\n    }}\n'
                + "".join(f'    attr {{\n      key: "{k}"\n      value {{\n        b: {"true" if k == flag else "false"}\n      }}\n    }}\n'
                          for k in ("transpose_a", "transpose_b")) + "  }\n")

    out = []
    for layer, x in acts.items():
        g = f"loss/gradients/train_model/{layer}"
        dy = f"{g}/add_grad/Reshape"
        out.append(node(f"{g}/MatMul_grad/MatMul", dy, f"model/{layer}/w/read", "transpose_b"))
        out.append(node(f"{g}/MatMul_grad/MatMul_1", x, dy, "transpose_a"))
    return "".join(out)


@pytest.mark.parametrize("activation", ["tanh", "relu"])
def test_readers_skip_the_gradient_matmuls(tmp_path, activation):
    """A real export also holds the gradient sub-graph, whose MatMuls read the same weights: the readers classify only the
    forward pass (the reference's own graph carries these nodes, SURVEY §3.5)."""
    from ppo_cpp_b200 import core
    path = _graph(tmp_path, activation)
    text = open(path, encoding="latin-1").read()
    with open(path, "w", encoding="latin-1") as f:
        f.write(text.replace("graph_def {\n", "graph_def {\n" + _grad_matmuls(activation), 1))
    assert mg.parse_meta_txt(path).activation == activation
    assert core.meta_activation(path) == activation
    core.meta_parse(path)


EDITS = {  # hand edits of the writer's tanh file, each of which the readers must refuse
    "elu": ('    name: "model/Tanh_2"\n    op: "Tanh"\n', '    name: "model/Tanh_2"\n    op: "Elu"\n'),
    "mixed": ('    name: "train_model/Tanh_3"\n    op: "Tanh"\n', '    name: "train_model/Tanh_3"\n    op: "Relu"\n'),
    "pi_fc2": ('graph_def {\n', 'graph_def {\n  node {\n    name: "model/pi_fc2/w"\n    op: "VariableV2"\n  }\n'),
    # the first pair's reader missing in one scope (train_model's pi_fc1 reads a weight that is no variable's read)
    "reader_missing": ('    name: "train_model/pi_fc1/MatMul"\n    op: "MatMul"\n    input: "train_model/Tanh"\n    input: "model/pi_fc1/w/read"\n',
                       '    name: "train_model/pi_fc1/MatMul"\n    op: "MatMul"\n    input: "train_model/Tanh"\n    input: "train_model/pi_fc1/w"\n'),
    "head_from_fc0": ('    name: "model/pi/MatMul"\n    op: "MatMul"\n    input: "model/Tanh_2"\n',
                      '    name: "model/pi/MatMul"\n    op: "MatMul"\n    input: "model/Tanh"\n'),
}


@pytest.mark.parametrize("edit", sorted(EDITS))
def test_readers_reject_an_unknown_forward_pass(tmp_path, edit):
    from ppo_cpp_b200 import core
    path = _graph(tmp_path, "tanh")
    text = open(path, encoding="latin-1").read()
    old, new = EDITS[edit]
    assert text.count(old) == 1
    with open(path, "w", encoding="latin-1") as f:
        f.write(text.replace(old, new))
    with pytest.raises(ValueError):
        mg.parse_meta_txt(path)
    with pytest.raises(core.PPOError, match=r"\[-4\]"):
        core.meta_activation(path)
    with pytest.raises(core.PPOError, match=r"\[-4\]"):
        core.meta_parse(path)


# ------------------------------------------------------------------ GPU: forward paths
def _core(core_mod, monkeypatch, env=(), activation="relu", **kw):
    for e in env:
        monkeypatch.setenv(e, "1")
    c = core_mod.PPOCore(activation=activation, **kw)
    for e in env:
        monkeypatch.delenv(e)
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("h,n,paths", [(4, 3000, [((), "small"), (("PPO_DISABLE_SMALL",), "tile")]),
                                       (64, 3000, [((), "fused"), (("PPO_DISABLE_FUSED",), "tile")]),
                                       (256, 2048, [((), "wgemm"), (("PPO_DISABLE_WIDE",), "tile")])])
def test_policy_paths_vs_fp64_and_each_other(monkeypatch, h, n, paths):
    from ppo_cpp_b200 import core as core_mod
    h2 = 5 if h == 4 else h
    rng = np.random.default_rng(40 + h)
    p = rand_params(rng, h, h2)
    obs = (2.0 * rng.standard_normal((n, 18))).astype(np.float32)
    eps = rng.standard_normal((n, 18)).astype(np.float32)
    mu64, v64 = forward_ref(p, obs, "relu", h, h2)
    outs = []
    for env, marker in paths:
        c = _core(core_mod, monkeypatch, env, hidden1=h, hidden2=h2, n_envs=n, n_steps=8, nminibatches=1)
        assert c.activation == "relu"
        c.set_tensor("params", p)
        assert marker in c.kernel_family("policy"), c.kernel_family("policy")
        a, v, nlp = c.policy_step(obs, eps)
        outs.append((a, v, nlp, c.policy_value(obs), c.policy_mean(obs)))
        c.close()
        assert rel_err(outs[-1][3], v64) < TOL and rel_err(outs[-1][4], mu64) < TOL, marker
        assert rel_err(v, v64) < TOL
    if h != 256:  # the fp32 CUDA-core paths compute the same operations in the same order
        for x, y in zip(outs[0], outs[1]):
            assert np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("h1,h2,n_envs,n_steps", [(64, 64, 4096, 16), (4, 5, 1, 256), (4, 5, 77, 40)])
def test_rollout_persistent_equals_stepwise_relu(monkeypatch, h1, h2, n_envs, n_steps):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(5)
    p = rand_params(rng, h1, h2)
    res = []
    for env in ((), ("PPO_DISABLE_PERSISTENT",)):
        c = _core(core_mod, monkeypatch, env, hidden1=h1, hidden2=h2, n_envs=n_envs, n_steps=n_steps, nminibatches=1, noptepochs=1, seed=11)
        c.set_tensor("params", p)
        assert ("persistent" in c.kernel_family("rollout")) == (not env)
        c.synth_env_reset()
        c.rollout_synthetic()
        c.rollout_synthetic()
        res.append({n: c.rollout_get(n) for n in ("obs", "actions", "values", "neglogpacs", "dones", "returns")})
        c.close()
    a, b = res
    assert np.array_equal(a["dones"], b["dones"])
    for name in ("obs", "actions", "values", "neglogpacs", "returns"):
        assert rel_err(a[name], b[name]) < 2e-5, name
    assert np.array_equal(a["actions"][:n_envs], b["actions"][:n_envs])  # first step: same observation, same forward pass


@pytest.mark.gpu
def test_host_env_rollout_equals_stepwise_relu(monkeypatch):
    from ppo_cpp_b200 import core as core_mod
    _, flat = load_weights("graph_4_5_init.npz")
    n_envs, n_steps, seed = 64, 24, 8
    lib = ol.load()
    res = []
    for disable in (False, True):
        if disable:
            monkeypatch.setenv("PPO_DISABLE_HOST_PERSISTENT", "1")
        env = lib.oracle_synth_env_create(n_envs, 18, seed ^ 0x1234, 0)
        obs, rew, done = np.zeros((n_envs, 18), np.float32), np.zeros(n_envs, np.float32), np.zeros(n_envs, np.float32)
        c = core_mod.PPOCore(activation="relu", n_envs=n_envs, n_steps=n_steps, nminibatches=4, noptepochs=1, seed=seed)
        c.set_tensor("params", flat)
        lib.oracle_synth_env_reset(env, obs)
        c.runner_reset(obs)

        def step(t, act):
            lib.oracle_synth_env_step(env, np.ascontiguousarray(act), obs, rew, done)
            return obs, rew, done

        c.runner_rollout_host(step)
        res.append({n: c.rollout_get(n) for n in ("obs", "actions", "values", "neglogpacs", "returns", "dones")})
        c.close()
        lib.oracle_synth_env_destroy(env)
        monkeypatch.delenv("PPO_DISABLE_HOST_PERSISTENT", raising=False)
    for name in res[0]:
        assert np.array_equal(res[0][name], res[1][name]), name


# ------------------------------------------------------------------ GPU: loss + gradient of every family
FAMILIES = [  # (h, B, env switch, family marker, fixtures)
    (4, 2048, None, "small", ("random", "ties")),
    (64, 1000, "PPO_DISABLE_UMMA", "fused", ("random", "ties")),
    (64, 1000, "PPO_DISABLE_FUSED", "tile", ("random", "ties")),
    (64, 4096, None, "tcgen05", ("random", "ties", "range")),
    (256, 1000, None, "tcgen05", ("random", "ties", "range")),
]


@pytest.mark.gpu
@pytest.mark.parametrize("h,B,env,fam,fixtures", FAMILIES)
def test_loss_grad_relu_every_family_vs_fp64(monkeypatch, h, B, env, fam, fixtures):
    from ppo_cpp_b200 import core as core_mod
    h2 = 5 if h == 4 else h
    rng = np.random.default_rng(200 + h + B)
    sl = tensor_slices(h, h2)
    c = _core(core_mod, monkeypatch, (env,) if env else (), hidden1=h, hidden2=h2, n_envs=4, n_steps=8, nminibatches=4)
    assert fam in c.kernel_family("train"), c.kernel_family("train")
    for fixture in fixtures:
        p = {"random": rand_params, "ties": tie_params}[fixture](rng, h, h2) if fixture != "range" else range_params(rng, h)
        c.set_tensor("params", p)
        obs, act, adv, ret, old_nlp, old_v = batch(rng, p, "relu", h, h2, B)
        if fixture == "range":
            lay, _ = _layout(h, h2)
            x = np.maximum(obs.astype(np.float64) @ p[lay[0][0]:lay[0][0] + 18 * h].reshape(18, h) + p[lay[1][0]:lay[1][0] + h], 0)
            h2v = np.maximum(x @ p[lay[4][0]:lay[4][0] + h * h].reshape(h, h) + p[lay[5][0]:lay[5][0] + h], 0)
            assert h2v.max() > 1000 and 0 < np.min(h2v[h2v > 0]) < 1e-3, (h2v.max(), np.min(h2v[h2v > 0]))
        g, l = c.loss_grad(obs, act, adv, ret, old_nlp, old_v, 0.2)
        g64, l64 = loss_grad_ref(p, obs, act, adv, ret, old_nlp, old_v, 0.2, "relu", h, h2)
        for t in range(13):
            assert rel_err(g[sl[t]], g64[sl[t]]) < TOL, (fixture, t, rel_err(g[sl[t]], g64[sl[t]]))
        assert np.allclose(l[:4], l64[:4], rtol=TOL, atol=1e-7), (fixture, l, l64)
    c.close()


# ------------------------------------------------------------------ GPU: whole updates against an fp64 learner
def learner_ref(flat, bufs, perms, nmb, lr, cr, h1, h2, clip=0.5, b1=0.9, b2=0.999, eps=1e-5):
    _, P = _layout(h1, h2)
    p = flat.astype(np.float64).copy()
    m, v = np.zeros(P), np.zeros(P)
    b1p, b2p = b1, b2
    nb = bufs["obs"].shape[0]
    Bm = nb // nmb
    rows = []
    for perm in perms:
        src = np.empty_like(perm)
        src[perm] = np.arange(nb)
        for k in range(nmb):
            idx = src[k * Bm:(k + 1) * Bm]
            ret, val = bufs["returns"][idx, 0], bufs["values"][idx, 0]
            a = ret.astype(np.float64) - val
            adv = (a - a.mean()) / (np.sqrt(((a - a.mean()) ** 2).mean()) + 1e-8)
            g, l = loss_grad_ref(p, bufs["obs"][idx], bufs["actions"][idx], adv, ret, bufs["neglogpacs"][idx, 0], val, cr, "relu", h1, h2)
            rows.append(l)
            gn = np.sqrt((g * g).sum())
            g = g * clip * min(1.0 / gn, 1.0 / clip)
            m += (g - m) * (1 - b1)
            v += (g * g - v) * (1 - b2)
            p[:P] -= lr * np.sqrt(1 - b2p) / (1 - b1p) * m / (np.sqrt(v) + eps)
            b1p *= b1
            b2p *= b2
    return p, np.mean(rows, axis=0)


@pytest.mark.gpu
@pytest.mark.parametrize("h1,h2,n_envs,n_steps,nmb,epochs,fam", [(4, 5, 1, 2048, 32, 2, "small"), (64, 64, 1024, 16, 2, 2, "persistent"),
                                                                  (256, 256, 128, 32, 1, 1, "tcgen05")])
def test_train_update_relu_vs_fp64_learner(h1, h2, n_envs, n_steps, nmb, epochs, fam):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(21)
    flat = load_weights("graph_4_5_init.npz")[1] if h1 == 4 else rand_params(rng, h1, h2)
    c = core_mod.PPOCore(activation="relu", hidden1=h1, hidden2=h2, n_envs=n_envs, n_steps=n_steps, nminibatches=nmb, noptepochs=epochs,
                         ent_coef=ENT, seed=9)
    c.set_tensor("params", flat)
    assert fam in c.kernel_family("train"), c.kernel_family("train")
    c.synth_env_reset()
    c.rollout_synthetic()
    bufs = {n: c.rollout_get(n) for n in ("obs", "actions", "returns", "values", "neglogpacs")}
    c.shuffle_seed(42)
    losses = c.train_update(3.9e-4, 0.2)
    perms = [c.train_get_permutation(e) for e in range(epochs)]
    got = c.get_tensor("params")
    c.close()
    p64, want = learner_ref(flat, bufs, perms, nmb, 3.9e-4, 0.2, h1, h2)
    _, P = _layout(h1, h2)
    moved = np.abs(p64[:P] - flat[:P]).max()
    assert np.abs(got[:P] - p64[:P]).max() < max(5e-4, 4e-5 * epochs * nmb) * moved
    assert np.abs(got[:P] - p64[:P]).max() < 1e-6 * max(1.0, np.abs(p64[:P]).max()) * epochs * nmb
    assert np.allclose(losses[:4], want[:4], rtol=2e-5, atol=1e-6), (losses, want)


# ------------------------------------------------------------------ GPU: selection, switching, the CLI
@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(hidden1=64, hidden2=64, n_envs=2048, n_steps=128, nminibatches=32),   # C3
                                dict(hidden1=256, hidden2=256, n_envs=1024, n_steps=64, nminibatches=4),   # the C4 shard
                                dict(n_envs=4096, n_steps=64, nminibatches=32),                              # c1x4096
                                dict(n_envs=1, n_steps=2048, nminibatches=32)])                              # C1
def test_relu_selects_the_same_families(kw):
    from ppo_cpp_b200 import core as core_mod
    names = []
    for act in ("tanh", "relu"):
        c = core_mod.PPOCore(activation=act, **kw)
        names.append([c.kernel_family(w) for w in ("train", "policy", "rollout")])
        c.close()
    assert names[0] == names[1]


@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 4])
def test_set_activation_switches_like_fresh_cores(h):
    from ppo_cpp_b200 import core as core_mod
    """tanh -> relu -> tanh on one core: the same gradients as fresh cores, bit for bit, and each switch re-captures the
    update graph once (the first update also captures the shuffle graph, which does not depend on the activation)."""
    h2 = 5 if h == 4 else h
    kw = dict(hidden1=h, hidden2=h2, n_envs=256, n_steps=32, nminibatches=4, noptepochs=2, seed=4)
    rng = np.random.default_rng(6)
    p = rand_params(rng, h, h2)
    data = batch(rng, p, "relu", h, h2, 512)
    fresh = {}
    for act in ("tanh", "relu"):
        c = core_mod.PPOCore(activation=act, **kw)
        c.set_tensor("params", p)
        fresh[act] = c.loss_grad(*data, 0.2)
        c.close()
    c = core_mod.PPOCore(**kw)
    c.synth_env_reset()
    seen = []
    for act in ("tanh", "relu", "tanh"):
        c.activation = act
        assert c.activation == act
        c.set_tensor("params", p)
        g, l = c.loss_grad(*data, 0.2)
        assert np.array_equal(g, fresh[act][0]) and np.array_equal(l, fresh[act][1]), act
        c.rollout_synthetic()
        before = c.graph_builds()
        c.train_update(3e-4, 0.2)
        c.train_update(3e-4, 0.2)
        seen.append(c.graph_builds() - before)
    c.close()
    assert seen[0] >= 1 and seen[1:] == [1, 1], seen
    with pytest.raises(ValueError):
        core_mod.PPOCore(activation="elu")


@pytest.mark.gpu
def test_cli_relu_round_trip(tmp_path):
    host = os.path.join(ROOT, "ppo_cpp_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    exe = os.path.join(host, "bin", "ppo_cpp")
    common = ["--threads", "2", "--seed", "5"]
    r = subprocess.run([exe, "-d", str(tmp_path / "exp"), "--id", "r0", "--activation", "relu", "--hidden", "64,64", "--steps", "4096",
                        "--num_epochs", "2", "--batch_steps", "1024", "--saves", "1", *common], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    ck = tmp_path / "exp" / "checkpoints" / "r0"
    side = [f for f in os.listdir(ck) if f.endswith(".json")]
    assert side and all('"activation": "relu"' in open(ck / f).read() or '"activation":"relu"' in open(ck / f).read() for f in side), side
    prefix = str(ck / side[0][:-len(".json")])
    r = subprocess.run([exe, "-p", prefix, "--duration", "0.3", *common], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "episode_reward" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    r = subprocess.run([exe, "-p", prefix, "--duration", "0.3", "--activation", "tanh", *common], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "contradicts the checkpoint" in r.stderr
    graph = _graph(tmp_path, "relu")
    r = subprocess.run([exe, "-g", graph, "--activation", "tanh", *common], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "contradicts the graph" in r.stderr
