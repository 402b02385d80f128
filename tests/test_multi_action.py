"""MultiDiscrete and MultiBinary action spaces: Stable-Baselines' MultiCategoricalProbabilityDistribution and
BernoulliProbabilityDistribution heads (ppo_action_space MULTI_DISCRETE / MULTI_BINARY).

The reference is an fp64 PyTorch autograd restatement of the PPO2 loss with either head: for MultiDiscrete one categorical per
slice of the logits (neglogp from log_softmax, the entropy as Stable-Baselines writes it), summed over the slices; for MultiBinary
TensorFlow's sigmoid_cross_entropy_with_logits in its where-form, the entropy sce(l, sigmoid(l)) differentiated through the labels.
CPU tests: both graph readers on the writer's files and hand edits, the layout and the checkpoint order, and the host bandit
modes.  GPU tests (the F and T families, tanh and ReLU): policy steps with given uniforms and with Philox noise, MultiDiscrete([n])
against Discrete(n), loss and gradients, whole updates against an fp64 learner, the host-env protocol, family selection,
checkpoints and graphs, and the CLI.  No real Stable-Baselines MultiDiscrete or MultiBinary export is available, so the reader rule
is checked against the writer's files and hand edits."""
import os
import subprocess
from functools import partial

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_err
from ppo_cpp_b200 import meta_graph as mg
from test_abi_cpu import _parse_bundle_index
from test_vf_clip_and_schedules import _tf_clip, _tf_max, learner_ref, value_loss

TOL = 1e-5
ENT = 0.01
O = 6
NVEC = [3, 5, 2]  # slices that straddle the Philox blocks of 4, a tail of 2
NB = 6            # MultiBinary width (a tail of 2)
SPACES = {"multi_discrete": dict(nvec=NVEC), "multi_binary": dict(act_dim=NB)}
FT = [((), "fused"), (("PPO_DISABLE_FUSED",), "tile")]


def width(space):
    return sum(NVEC) if space == "multi_discrete" else NB


def slices(space):
    if space == "multi_binary":
        return None
    off = np.concatenate([[0], np.cumsum(NVEC)])
    return [(int(off[i]), int(off[i + 1])) for i in range(len(NVEC))]


# ------------------------------------------------------------------ layout and the fp64 reference
def layout(space, h1, h2):
    lay = mg.param_layout(O, width(space), h1, h2, action_space=space)
    order = [t for t in mg.TENSOR_ORDER[:mg.N_TRAINABLE_TENSORS] if t != mg.LOGSTD]
    return [lay[t] for t in order], lay["model/q/w"][0], lay["__total__"][0]


def rand_params(rng, space, h1, h2, head_scale=1.0):
    _, _, Pq = layout(space, h1, h2)
    p = (rng.standard_normal(Pq) * min(0.3, 1.5 / np.sqrt(max(h1, h2)))).astype(np.float32)
    off = mg.param_layout(O, width(space), h1, h2, action_space=space)["model/pi/w"][0]
    p[off:off + h2 * width(space)] *= 4.0 * head_scale
    return p


def forward_ref(params, obs, activation, space, h1, h2):
    lay, _, _ = layout(space, h1, h2)
    t = [params.astype(np.float64)[off:off + int(np.prod(s))].reshape(s) for off, s in lay]
    f = np.tanh if activation == "tanh" else (lambda z: np.maximum(z, 0.0))
    x = obs.astype(np.float64)
    logits = f(f(x @ t[0] + t[1]) @ t[4] + t[5]) @ t[10] + t[11]
    v = (f(f(x @ t[2] + t[3]) @ t[6] + t[7]) @ t[8] + t[9])[:, 0]
    return logits, v


def sce(l, z):
    """TF's sigmoid_cross_entropy_with_logits as it builds it: where(l >= 0, l, 0) - l z + log1p(exp(where(l >= 0, -l, l)))."""
    pos = l >= 0
    return torch.where(pos, l, torch.zeros_like(l)) - l * z + torch.log1p(torch.exp(torch.where(pos, -l, l)))


def nlp_ent(logits, act, space):
    """Per-sample neglogp of act and entropy of the head, torch fp64."""
    if space == "multi_binary":
        return sce(logits, act).sum(1), sce(logits, torch.sigmoid(logits)).sum(1)
    nlp, ent = 0.0, 0.0
    for i, (a, b) in enumerate(slices(space)):
        li = logits[:, a:b]
        nlp = nlp - torch.log_softmax(li, 1).gather(1, act[:, i:i + 1].long())[:, 0]
        a0 = li - li.max(1, keepdim=True)[0]
        z = torch.exp(a0).sum(1, keepdim=True)
        ent = ent + ((torch.exp(a0) / z) * (torch.log(z) - a0)).sum(1)
    return nlp, ent


def neglogp_np(logits, act, space):
    n, _ = nlp_ent(torch.tensor(logits), torch.tensor(np.asarray(act, np.float64)), space)
    return n.numpy()


def loss_grad_ref(params, obs, act, adv, ret, old_nlp, old_v, cr, activation, space, h1, h2, ent_coef=ENT, vf_coef=0.5, vf="shared", cr_vf=0.0):
    lay, P, _ = layout(space, h1, h2)
    p = torch.tensor(np.asarray(params[:P], np.float64), requires_grad=True)
    pi0w, pi0b, vf0w, vf0b, pi1w, pi1b, vf1w, vf1b, vfw, vfb, piw, pib = [p[off:off + int(np.prod(s))].reshape(s) for off, s in lay]
    f = torch.tanh if activation == "tanh" else torch.relu
    x = torch.tensor(np.asarray(obs, np.float64))
    a = torch.tensor(np.asarray(act, np.float64))
    adv, R, onl, ov = (torch.tensor(np.asarray(z, np.float64).ravel()) for z in (adv, ret, old_nlp, old_v))
    logits = f(f(x @ pi0w + pi0b) @ pi1w + pi1b) @ piw + pib
    v = (f(f(x @ vf0w + vf0b) @ vf1w + vf1b) @ vfw + vfb)[:, 0]
    nlp, ent = nlp_ent(logits, a, space)
    ratio = torch.exp(onl - nlp)
    pg = _tf_max(-adv * ratio, -adv * _tf_clip(ratio, torch.tensor(1.0 - cr, dtype=torch.float64),
                                                torch.tensor(1.0 + cr, dtype=torch.float64))).mean()
    vfl = 0.5 * value_loss(v, ov, R, vf, cr, cr_vf).mean()
    ent = ent.mean()
    loss = pg - ent * ent_coef + vfl * vf_coef
    loss.backward()
    with torch.no_grad():
        kl = 0.5 * ((nlp - onl) ** 2).mean()
        cf = ((ratio - 1.0).abs() > cr).double().mean()
    return p.grad.numpy().copy(), np.array([pg.item(), vfl.item(), ent.item(), kl.item(), cf.item()])


def sample_actions(rng, logits, space):
    if space == "multi_binary":
        return (rng.uniform(size=logits.shape) < 1.0 / (1.0 + np.exp(-logits))).astype(np.float32)
    cols = []
    for a, b in slices(space):
        q = np.exp(logits[:, a:b] - logits[:, a:b].max(1, keepdims=True))
        q /= q.sum(1, keepdims=True)
        cols.append([rng.choice(b - a, p=r) for r in q])
    return np.array(cols, np.float32).T


def batch(rng, params, activation, space, h1, h2, B):
    obs = rng.standard_normal((B, O)).astype(np.float32)
    logits, v = forward_ref(params, obs, activation, space, h1, h2)
    act = sample_actions(rng, logits, space)
    old_nlp = (neglogp_np(logits, act, space) + 0.1 * rng.standard_normal(B)).astype(np.float32)
    old_v = (v + 0.3 * rng.standard_normal(B)).astype(np.float32)
    ret = (v + 0.3 + 0.5 * rng.standard_normal(B)).astype(np.float32)
    adv = rng.standard_normal(B).astype(np.float32)
    return obs, act, adv, ret, old_nlp, old_v


def uniform_fixture(rng, logits, space):
    """Uniforms whose sampled action fp32 rounding cannot change: for MultiDiscrete each slice's Gumbel maximum is at least 1e-3
    above its runner-up, with u = 0 (never taken) at the first logit of slice 1 in every tenth row; for MultiBinary every u is at
    least 1e-3 away from sigmoid(l).  Returns (u, the actions they give)."""
    B, A = logits.shape
    u = rng.uniform(0.0, 1.0, (B, A))
    if space == "multi_binary":
        s = 1.0 / (1.0 + np.exp(-logits))
        for _ in range(100):
            bad = np.abs(u - s) < 1e-3
            if not bad.any():
                break
            u[bad] = rng.uniform(0.0, 1.0, int(bad.sum()))
        return u.astype(np.float32), (u < s).astype(np.float32)
    u[::10, slices(space)[1][0]] = 0.0
    acts = np.zeros((B, len(NVEC)))
    for i, (a, b) in enumerate(slices(space)):
        for _ in range(100):
            with np.errstate(divide="ignore"):
                g = logits[:, a:b] - np.log(-np.log(u[:, a:b]))
            srt = np.sort(g, 1)
            bad = srt[:, -1] - srt[:, -2] < 1e-3
            if not bad.any():
                break
            u[bad, a:b] = rng.uniform(0.0, 1.0, (int(bad.sum()), b - a))
        acts[:, i] = np.argmax(g, 1)
    return u.astype(np.float32), acts.astype(np.float32)


def deterministic_ref(logits, space):
    if space == "multi_binary":
        return (logits > 0).astype(np.float32)  # round(sigmoid(l)) with ties to even: l = 0 gives 0
    return np.stack([np.argmax(logits[:, a:b], 1) for a, b in slices(space)], 1).astype(np.float32)


# ------------------------------------------------------------------ CPU: the graph readers and the writer
def _tensors(space, h1=4, h2=5):
    rng = np.random.default_rng(1)
    return {name: rng.standard_normal(s).astype(np.float32) for name, (off, s) in mg.param_layout(O, width(space), h1, h2).items() if name != "__total__"}


def _graph(tmp_path, space, activation=None, nvec=None, name=None):
    path = str(tmp_path / (name or f"g_{space}.meta.txt"))
    if space == "multi_discrete" and nvec is None:
        nvec = NVEC
    mg.write_meta_txt(path, _tensors(space), ent_coef=ENT, action_space=space, activation=activation, nvec=nvec)
    return path


@pytest.mark.parametrize("activation", [None, "relu"])
@pytest.mark.parametrize("dtype", ["DT_INT32", "DT_INT64"])
@pytest.mark.parametrize("space", sorted(SPACES))
def test_readers_classify_the_new_spaces(tmp_path, space, dtype, activation):
    from ppo_cpp_b200 import core
    path = _graph(tmp_path, space, activation=activation)
    text = open(path, encoding="latin-1").read()
    assert mg.LOGSTD not in text and "loss/action_ph" in text
    for t in ("DT_INT32\n      }\n    }\n    attr {\n      key: \"shape\"", "DT_INT64\n      }\n    }\n    attr {\n      key: \"shape\""):
        text = text.replace(t, dtype + t[8:])
    with open(path, "w", encoding="latin-1") as f:
        f.write(text)
    want_nvec = NVEC if space == "multi_discrete" else [2] * NB
    info = mg.parse_meta_txt(path)
    assert info.action_space == mg.meta_action_space(path) == core.meta_action_space(path) == space
    assert info.nvec == core.meta_action_nvec(path) == want_nvec
    assert core.meta_activation(path) == (activation or "tanh")
    cinfo, params = core.meta_parse(path)
    lay = mg.param_layout(O, width(space), 4, 5, action_space=space)
    assert (cinfo.obs_dim, cinfo.act_dim) == (O, width(space))
    assert cinfo.n_params_total == lay["__total__"][0] and cinfo.n_params_trainable == lay["model/q/w"][0]
    np.testing.assert_array_equal(params, info.flat_params())


def test_readers_nvec_of_the_old_spaces(tmp_path):
    from ppo_cpp_b200 import core
    for space, want in (("discrete", [width("multi_binary")]), ("box", None)):
        path = str(tmp_path / f"{space}.meta.txt")
        mg.write_meta_txt(path, _tensors("multi_binary"), action_space=space)
        assert mg.parse_meta_txt(path).nvec == want
        if want is None:
            with pytest.raises(core.PPOError, match=r"\[-1\]"):
                core.meta_action_nvec(path)
        else:
            assert core.meta_action_nvec(path) == want
    with pytest.raises(ValueError):
        mg.write_meta_txt(str(tmp_path / "x.meta.txt"), _tensors("multi_discrete"), action_space="multi_discrete", nvec=[3, 5])  # sums to 8, not 10
    with pytest.raises(ValueError):
        mg.write_meta_txt(str(tmp_path / "x.meta.txt"), _tensors("multi_discrete"), action_space="multi_binary", nvec=NVEC)


_SPLIT_IN = 'input: "model/pi/add"\n    input: "model/split/size_splits"'


def _sizes(v):
    return mg._escape(np.asarray(v, "<i4").tobytes())


EDITS = {  # hand edits both readers must refuse: (space, old, new, the node the error names)
    "sizes_do_not_sum_to_width": ("multi_discrete", _sizes(NVEC), _sizes([3, 4, 2]), "model/split"),
    "split_count_is_not_k": ("multi_discrete", "size: -1\n          }\n          dim {\n            size: 3", "size: -1\n          }\n          dim {\n            size: 2", "model/split"),
    "split_reads_another_tensor": ("multi_discrete", _SPLIT_IN, _SPLIT_IN.replace("model/pi/add", "model/vf/add"), "loss/action_ph"),
    "k_is_not_width_without_split": ("multi_binary", "size: -1\n          }\n          dim {\n            size: 6", "size: -1\n          }\n          dim {\n            size: 5", "model/Sigmoid"),
    "no_bernoulli_head": ("multi_binary", 'name: "model/Sigmoid"\n    op: "Sigmoid"', 'name: "model/Sigmoid"\n    op: "Tanh"', "loss/action_ph"),
    "float_rank_2_without_logstd": ("multi_binary", "type: DT_INT32", "type: DT_FLOAT", "loss/action_ph"),
}


@pytest.mark.parametrize("edit", sorted(EDITS))
def test_readers_reject_hand_edits(tmp_path, edit):
    from ppo_cpp_b200 import core
    space, old, new, node = EDITS[edit]
    path = _graph(tmp_path, space)
    text = open(path, encoding="latin-1").read()
    assert text.count(old) == 1, edit
    with open(path, "w", encoding="latin-1") as f:
        f.write(text.replace(old, new))
    with pytest.raises(ValueError, match=node):
        mg.parse_meta_txt(path)
    for fn in (core.meta_action_space, core.meta_parse, core.meta_action_nvec):
        with pytest.raises(core.PPOError, match=rf"\[-4\].*{node}"):
            fn(path)


@pytest.mark.parametrize("space", sorted(SPACES))
def test_param_layout_and_index_round_trip(tmp_path, space):
    import ctypes as C
    from ppo_cpp_b200 import _lib
    A = width(space)
    lay, disc = mg.param_layout(O, A, 8, 8, action_space=space), mg.param_layout(O, A, 8, 8, action_space="discrete")
    assert lay == disc  # the same layout as a categorical head over the same logits: no logstd
    shapes = {t: s for t, (o, s) in lay.items() if t != "__total__"}
    payload = {t: np.random.default_rng(2).standard_normal(s).astype(np.float32) for t, s in shapes.items()}
    raw = np.concatenate([payload[t].ravel() for t in mg.CKPT_ORDER if t in payload])
    raw.tofile(tmp_path / "c.data-00000-of-00001")
    got = mg.read_checkpoint_data(str(tmp_path / "c.data-00000-of-00001"), shapes)
    assert list(got) == [t for t in mg.CKPT_ORDER if t != mg.LOGSTD]
    for t in shapes:
        np.testing.assert_array_equal(got[t], payload[t])
    lib = _lib.load()
    fp = raw.ctypes.data_as(C.POINTER(C.c_float))
    assert lib.ppo_checkpoint_write_index_ex(str(tmp_path / "c").encode(), _lib.PPO_ACTION_DISCRETE, O, A, 8, 8, fp, raw.size) == 0
    ent = _parse_bundle_index(open(tmp_path / "c.index", "rb").read())
    assert list(ent)[1:] == list(got) and all(tuple(ent[t]["shape"]) == shapes[t] for t in got)


@pytest.mark.parametrize("mode", ["md", "mb"])
def test_host_bandit_modes(tmp_path, mode):
    """The CLI's bandit_md / bandit_mb envs: the action space and width PPO2 sees, and the reward of a perfect and of a wrong policy."""
    src = tmp_path / "b.cpp"
    md = mode == "md"
    src.write_text('#include "env_bandit.hpp"\n#include <cstdio>\nint main() {\n'
                   f'  BanditEnv e(7, 0, 4, BanditEnv::{"MULTI_DISCRETE" if md else "MULTI_BINARY"});\n  Mat obs = e.reset();\n'
                   f'  int ok = e.get_action_space() == Env::{"SPACE_MULTI_DISCRETE" if md else "SPACE_MULTI_BINARY"}() && action_width(e) == {2 if md else 4}'
                   f' && e.get_action_space_size() == {7 if md else 4} && e.get_action_space_nvec() == std::vector<int>{{{"4, 3" if md else ""}}};\n'
                   '  float good = 0, bad = 0, dones = 0;\n  int seen = 0;\n  for (int t = 0; t < 64; ++t) {\n    int c = 0;\n'
                   + ('    for (int k = 0; k < 4; ++k) if (obs(0, k) > 0.5f) c = k;\n    seen |= 1 << c;\n'
                      '    Mat a(1, 2); a(0, 0) = (float)((c + 1 + (t & 1)) % 4); a(0, 1) = (float)((c + (t & 1)) % 3);\n' if md else
                      '    for (int k = 0; k < 4; ++k) c |= (obs(0, k) > 0.5f ? 1 : 0) << k;\n    seen |= 1 << c;\n'
                      '    Mat a(1, 4); for (int k = 0; k < 4; ++k) a(0, k) = (float)(((c >> k) & 1) ^ (t & 1));\n')
                   + '    auto r = e.step(a);\n    (t & 1 ? bad : good) += r[1](0, 0); dones += r[2](0, 0); obs = r[0];\n  }\n'
                   '  std::printf("%d %g %g %g %d\\n", ok, good, bad, dones, __builtin_popcount(seen));\n  return 0;\n}\n')
    exe = tmp_path / "b"
    subprocess.run(["g++", "-std=c++14", "-O1", "-I", os.path.join(ROOT, "ppo_cpp_b200", "host"), "-o", str(exe), str(src)], check=True)
    ok, good, bad, dones, seen = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert (int(ok), float(good), float(bad), float(dones)) == (1, 32.0, 0.0, 4.0)
    assert int(seen) >= (4 if md else 12)  # the contexts drawn cover the space


# ------------------------------------------------------------------ GPU
def _core(core_mod, monkeypatch, space, env=(), **kw):
    for e in env:
        monkeypatch.setenv(e, "1")
    kw.setdefault("obs_dim", O)
    kw = {**SPACES[space], **kw}
    c = core_mod.PPOCore(action_space=space, **kw)
    for e in env:
        monkeypatch.delenv(e)
    assert c.action_space == space
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ["tanh", "relu"])
@pytest.mark.parametrize("env,fam", FT)
@pytest.mark.parametrize("space", sorted(SPACES))
def test_policy_step_with_given_uniforms_vs_fp64(monkeypatch, space, env, fam, activation):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(3)
    B, A = 3000, width(space)
    p = rand_params(rng, space, 64, 64)
    obs = rng.standard_normal((B, O)).astype(np.float32)
    logits, v64 = forward_ref(p, obs, activation, space, 64, 64)
    u, want = uniform_fixture(rng, logits, space)
    c = _core(core_mod, monkeypatch, space, env, activation=activation, hidden1=64, hidden2=64, n_envs=B, n_steps=2, nminibatches=1)
    assert fam in c.kernel_family("policy") and fam in c.kernel_family("train"), c.kernel_family("policy")
    assert c.nvec == (NVEC if space == "multi_discrete" else [2] * NB) and c.AW == want.shape[1]
    c.set_tensor("params", p)
    a, v, nlp = c.policy_step(obs, u)
    assert np.array_equal(a, want)
    if space == "multi_discrete":
        assert not np.any(a[::10, 1] == 0.0)  # u = 0 is never taken
    assert rel_err(nlp, neglogp_np(logits, want, space)) < TOL and rel_err(v, v64) < TOL
    det = c.policy_mean(obs)
    if space == "multi_discrete":
        sep = np.all([np.sort(logits[:, a_:b_], 1)[:, -1] - np.sort(logits[:, a_:b_], 1)[:, -2] > 1e-4 for a_, b_ in slices(space)], 0)
    else:
        sep = np.all(np.abs(logits) > 1e-4, 1)
    assert np.array_equal(det[sep], deterministic_ref(logits, space)[sep])
    # ties: equal logits in a slice give its first index; l = 0 gives bit 0; nlp is the sum of log(n_i) / n log 2
    q = p.copy()
    lay = mg.param_layout(O, A, 64, 64, action_space=space)
    q[lay["model/pi/w"][0]:lay["model/pi/w"][0] + 64 * A] = 0.0
    q[lay["model/pi/b"][0]:lay["model/pi/b"][0] + A] = 0.0 if space == "multi_binary" else 0.25
    c.set_tensor("params", q)
    a, _, nlp = c.policy_step(obs[:64], np.full((64, A), 0.5, np.float32) if space == "multi_discrete" else np.full((64, A), 0.75, np.float32))
    assert np.all(a == 0.0) and np.all(c.policy_mean(obs[:64]) == 0.0)
    assert np.allclose(nlp, np.log(NVEC).sum() if space == "multi_discrete" else NB * np.log(2.0), rtol=1e-6)
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env,fam", FT)
def test_multi_discrete_of_one_slice_is_discrete(monkeypatch, env, fam):
    """MultiDiscrete([n]) and Discrete(n) with the same seed and weights: the Philox policy step, ppo_loss_grad and a whole update
    are bit-identical."""
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(17)
    n, h, n_envs, n_steps = 7, 64, 128, 16
    kw = dict(obs_dim=O, act_dim=n, hidden1=h, hidden2=h, n_envs=n_envs, n_steps=n_steps, nminibatches=4, noptepochs=2, ent_coef=ENT, seed=5)
    p = (rng.standard_normal(mg.param_layout(O, n, h, h, action_space="discrete")["__total__"][0]) * 0.2).astype(np.float32)
    obs = rng.standard_normal((n_envs, O)).astype(np.float32)
    raw = rng.standard_normal((n_steps, n_envs, O)).astype(np.float32)
    rew = rng.standard_normal((n_steps, n_envs)).astype(np.float32)
    done = (rng.uniform(size=(n_steps, n_envs)) < 0.05).astype(np.float32)
    B = 500
    lg = (rng.standard_normal((B, O)).astype(np.float32), rng.integers(0, n, (B, 1)).astype(np.float32), rng.standard_normal(B),
          rng.standard_normal(B), rng.standard_normal(B) + 2.0, rng.standard_normal(B))
    out = []
    for space in ("discrete", "multi_discrete"):
        for e in env:
            monkeypatch.setenv(e, "1")
        c = core_mod.PPOCore(action_space=space, nvec=[n] if space == "multi_discrete" else None, **kw)
        for e in env:
            monkeypatch.delenv(e)
        assert fam in c.kernel_family("train")
        c.set_tensor("params", p)
        step = c.policy_step(obs)
        grads = c.loss_grad(*lg, 0.2)
        c.runner_reset(obs)
        c.runner_rollout_replay(raw, rew, done)
        c.shuffle_seed(3)
        losses = c.train_update(3e-4, 0.2)
        out.append((step, grads, losses, c.get_tensor("params"), c.get_tensor("adam_m")))
        c.close()
    for x, y in zip(out[0], out[1]):
        for xa, ya in zip(x if isinstance(x, tuple) else (x,), y if isinstance(y, tuple) else (y,)):
            assert np.array_equal(xa, ya)


@pytest.mark.gpu
@pytest.mark.parametrize("env,fam", FT)
@pytest.mark.parametrize("space", sorted(SPACES))
def test_philox_action_frequencies_match_the_model(monkeypatch, space, env, fam):
    """Every env sees the same observation: over 200 000 draws the index frequencies of each slice match its softmax and the
    slices are independent (MultiDiscrete), the bit frequencies match sigmoid(l) (MultiBinary); chi-square at a fixed seed."""
    from scipy import stats
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(4)
    B = 50000
    p = rand_params(rng, space, 64, 64, head_scale=0.3)
    obs = np.repeat(rng.standard_normal((1, O)).astype(np.float32), B, 0)
    logits, _ = forward_ref(p, obs[:1], "tanh", space, 64, 64)
    c = _core(core_mod, monkeypatch, space, env, hidden1=64, hidden2=64, n_envs=B, n_steps=2, nminibatches=1, seed=123)
    c.set_tensor("params", p)
    draws = []
    for _ in range(4):
        a, _, nlp = c.policy_step(obs)
        draws.append(a.copy())
        assert rel_err(nlp, neglogp_np(np.repeat(logits, B, 0), a, space)) < TOL
    c.close()
    assert not np.array_equal(draws[0], draws[1])  # the step counter advances the stream
    a = np.concatenate(draws)
    if space == "multi_binary":
        s = 1.0 / (1.0 + np.exp(-logits[0]))
        for j in range(NB):
            k = int(a[:, j].sum())
            assert stats.binomtest(k, len(a), s[j]).pvalue > 1e-3, (j, k / len(a), s[j])
        # independence of bits 0 and 1 (the same Philox word block)
        joint = np.array([[np.sum((a[:, 0] == x) & (a[:, 1] == y)) for y in (0, 1)] for x in (0, 1)])
        assert stats.chi2_contingency(joint)[1] > 1e-3
        return
    probs = []
    for i, (lo, hi) in enumerate(slices(space)):
        q = np.exp(logits[0, lo:hi] - logits[0, lo:hi].max())
        q /= q.sum()
        probs.append(q)
        counts = np.bincount(a[:, i].astype(int), minlength=hi - lo)
        assert stats.chisquare(counts, counts.sum() * q).pvalue > 1e-3, (i, counts / counts.sum(), q)
    joint = np.zeros((NVEC[0], NVEC[1]))
    np.add.at(joint, (a[:, 0].astype(int), a[:, 1].astype(int)), 1)
    assert stats.chi2_contingency(joint)[1] > 1e-3  # slices 0 and 1 share a Philox block: they must still be independent


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ["tanh", "relu"])
@pytest.mark.parametrize("space", sorted(SPACES))
def test_loss_grad_vs_fp64_and_f_equals_t(monkeypatch, space, activation):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(5)
    h = 64
    p = rand_params(rng, space, h, h)
    data = batch(rng, p, activation, space, h, h, 1000)
    lay, P, _ = layout(space, h, h)
    for vf, cr_vf in (("shared", None), ("separate", 0.15)):
        g64, l64 = loss_grad_ref(p, *data, 0.2, activation, space, h, h, vf=vf, cr_vf=cr_vf or 0.0)
        outs = []
        for env, fam in FT:
            c = _core(core_mod, monkeypatch, space, env, activation=activation, hidden1=h, hidden2=h, n_envs=4, n_steps=8, nminibatches=4, ent_coef=ENT)
            assert fam in c.kernel_family("train") and c.tensor_size("params_trainable") == P
            c.vf_clip = vf
            c.set_tensor("params", p)
            g, l = c.loss_grad(*data, 0.2, cliprange_vf=cr_vf)
            c.close()
            for t, (off, s) in enumerate(lay):
                sl = slice(off, off + int(np.prod(s)))
                assert rel_err(g[sl], g64[sl]) < TOL, (vf, fam, t, rel_err(g[sl], g64[sl]))
            assert np.allclose(l, l64, rtol=TOL, atol=1e-7), (vf, fam, l, l64)
            outs.append((g, l))
        assert rel_err(outs[0][0], outs[1][0]) < 2e-6 and np.allclose(outs[0][1], outs[1][1], rtol=2e-6, atol=1e-8)
    # the entropy term matters: without it the logits' gradient differs
    g0, _ = loss_grad_ref(p, *data, 0.2, activation, space, h, h, ent_coef=0.0)
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
@pytest.mark.parametrize("space", sorted(SPACES))
def test_train_update_vs_fp64_learner(monkeypatch, space, env, fam, activation, switch):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(21)
    h, n_envs, n_steps, nmb, epochs = 64, 128, 16, 4, 2
    flat = rand_params(rng, space, h, h)
    raw, rew, done = _replay_rollout(rng, n_envs, n_steps)
    c = _core(core_mod, monkeypatch, space, env + switch, activation=activation, hidden1=h, hidden2=h, n_envs=n_envs, n_steps=n_steps,
              nminibatches=nmb, noptepochs=epochs, ent_coef=ENT, seed=9)
    assert fam in c.kernel_family("train")
    c.set_tensor("params", flat)
    c.runner_reset(rng.standard_normal((n_envs, O)).astype(np.float32))
    c.runner_rollout_replay(raw, rew, done)
    bufs = {n: c.rollout_get(n) for n in ("obs", "actions", "returns", "values", "neglogpacs")}
    assert bufs["actions"].shape == (n_envs * n_steps, c.AW)
    c.shuffle_seed(42)
    losses = c.train_update(3.9e-4, 0.2)
    perms = [c.train_get_permutation(e) for e in range(epochs)]
    got = c.get_tensor("params")
    c.close()
    p64, want = learner_ref(flat, bufs, perms, nmb, 3.9e-4, 0.2, partial(loss_grad_ref, activation=activation, space=space, h1=h, h2=h))
    _, P, _ = layout(space, h, h)
    moved = np.abs(p64[:P] - flat[:P]).max()
    assert np.abs(got[:P] - p64[:P]).max() < max(5e-4, 4e-5 * epochs * nmb) * moved
    assert np.abs(got[:P] - p64[:P]).max() < 1e-6 * max(1.0, np.abs(p64[:P]).max()) * epochs * nmb
    assert np.allclose(losses, want, rtol=2e-5, atol=1e-6), (losses, want)


@pytest.mark.gpu
@pytest.mark.parametrize("env,fam", FT)
@pytest.mark.parametrize("space", sorted(SPACES))
def test_host_env_protocol_and_replay(monkeypatch, space, env, fam):
    """ppo_runner_rollout_replay, ppo_runner_rollout_host and the per-call act/observe loop store the same actions of the core's
    width, valid per column; invalid actions handed in are refused per column."""
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(8)
    n_envs, n_steps = 96, 12
    flat = rand_params(rng, space, 64, 64)
    obs0 = rng.standard_normal((n_envs, O)).astype(np.float32)
    raw, rew, done = _replay_rollout(rng, n_envs, n_steps)
    res = []
    for mode in ("replay", "host", "stepwise"):
        c = _core(core_mod, monkeypatch, space, env, hidden1=64, hidden2=64, n_envs=n_envs, n_steps=n_steps, nminibatches=4, seed=31)
        assert c.kernel_family("rollout") == "per-step kernels"
        c.set_tensor("params", flat)
        c.runner_reset(obs0)
        acts = np.zeros((n_steps, n_envs, c.AW), np.float32)
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
        if mode == "stepwise":
            nv = c.nvec
            good = res[0][1]["actions"]
            for col, bad in [(j, float(nv[j])) for j in range(len(nv))] + [(0, 0.5), (len(nv) - 1, -1.0)] + \
                            ([(NB - 1, 2.0)] if space == "multi_binary" else []):
                x = good.copy()
                x[5, col] = bad
                with pytest.raises(core_mod.PPOError, match=rf"\[-1\].*column {col}"):
                    c.rollout_set("actions", x)
                with pytest.raises(core_mod.PPOError, match=rf"\[-1\].*column {col}"):
                    c.loss_grad(res[0][1]["obs"][:16], x[:16], *(np.zeros(16),) * 4, 0.2)
            c.rollout_set("actions", good)
        c.close()
    acts = res[0][0]
    hi = np.array(NVEC if space == "multi_discrete" else [2] * NB) - 1
    assert np.array_equal(acts, np.round(acts)) and acts.min() >= 0 and np.all(acts.max((0, 1)) == hi)
    for a, bufs in res:
        assert np.array_equal(a, acts)
        assert np.array_equal(bufs["actions"].reshape(n_envs, n_steps, -1), acts.transpose(1, 0, 2))  # flat layout row = env * n_steps + t
        for k in bufs:
            assert np.array_equal(bufs[k], res[0][1][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("h1,h2", [(4, 5), (64, 64), (256, 256)])
@pytest.mark.parametrize("space", sorted(SPACES))
def test_family_selection_and_unsupported_paths(space, h1, h2):
    from ppo_cpp_b200 import core as core_mod
    kw = dict(obs_dim=18, hidden1=h1, hidden2=h2, n_envs=1024, n_steps=16, nminibatches=4)
    c = core_mod.PPOCore(action_space=space, **({"nvec": [6, 6, 6]} if space == "multi_discrete" else {"act_dim": 18}), **kw)
    assert c.tensor_size("params") == mg.param_layout(18, 18, h1, h2, action_space=space)["__total__"][0]
    fams = [c.kernel_family(w) for w in ("train", "policy", "rollout")]
    assert ("train_fused_kernel" in fams[0]) or ("train_tile_kernel" in fams[0]), fams
    assert ("policy_fused_kernel" in fams[1]) or ("policy_tile_kernel" in fams[1]), fams
    assert fams[2] == "per-step kernels"
    for fn in (c.synth_env_reset, c.rollout_synthetic, lambda: c.learn_update_synthetic(3e-4, 0.2)):
        with pytest.raises(core_mod.PPOError, match=r"\[-4\]"):
            fn()
    for name in (mg.LOGSTD, mg.LOGSTD + "/Adam"):
        with pytest.raises(core_mod.PPOError, match=r"\[-1\]"):
            c.tensor_size(name)
    c.close()
    # creation: MULTI_DISCRETE needs ppo_core_create_nvec; nvec must be positive and sum to act_dim <= 64
    import ctypes as C
    from ppo_cpp_b200 import _lib
    lib = _lib.load()
    d = _lib.CoreDesc()
    lib.ppo_core_desc_default(C.byref(d))
    d.obs_dim, d.act_dim, d.n_envs, d.n_steps, d.nminibatches = 18, 18, 8, 8, 2
    h = C.c_void_p()
    assert lib.ppo_core_create_ex(C.byref(d), _lib.PPO_ACTION_MULTI_DISCRETE, C.byref(h)) == -1
    for bad in ([6, 6, 5], [18, 0], [6, 6, 6, 1]):
        nv = np.array(bad, np.int32)
        assert lib.ppo_core_create_nvec(C.byref(d), nv.ctypes.data, nv.size, C.byref(h)) == -1, bad
    box = core_mod.PPOCore(obs_dim=18, act_dim=18, **{k: v for k, v in kw.items() if k != "obs_dim"})
    with pytest.raises(core_mod.PPOError, match=r"\[-1\]"):
        box.nvec
    box.close()


@pytest.mark.gpu
@pytest.mark.parametrize("space", sorted(SPACES))
def test_checkpoint_and_graph_round_trip(tmp_path, space):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(12)
    A = width(space)
    kw = dict(obs_dim=O, hidden1=64, hidden2=64, n_envs=8, n_steps=8, nminibatches=2)
    c = core_mod.PPOCore(action_space=space, **SPACES[space], **kw)
    lay = mg.param_layout(O, A, 64, 64, action_space=space)
    p = rand_params(rng, space, 64, 64)
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
    d = core_mod.PPOCore(action_space=space, **SPACES[space], **kw)
    d.load_checkpoint_data(prefix)
    assert np.array_equal(d.get_tensor("params"), p)
    d.close()
    t = {k: rng.standard_normal(s).astype(np.float32) for k, (o, s) in mg.param_layout(O, A, 64, 64).items() if k != "__total__"}
    g = str(tmp_path / "g.meta.txt")
    mg.write_meta_txt(g, t, ent_coef=ENT, action_space=space, nvec=NVEC if space == "multi_discrete" else None)
    c.load_meta_txt(g)
    assert np.array_equal(c.get_tensor("params"), mg.parse_meta_txt(g).flat_params())
    # a graph of another space, or of another nvec, is refused
    other = str(tmp_path / "o.meta.txt")
    if space == "multi_discrete":
        mg.write_meta_txt(other, t, ent_coef=ENT, action_space="multi_discrete", nvec=[5, 3, 2])
        with pytest.raises(core_mod.PPOError, match=r"\[-1\].*nvec"):
            c.load_meta_txt(other)
    for sp in ("discrete", "multi_binary" if space == "multi_discrete" else "multi_discrete"):
        mg.write_meta_txt(other, t, ent_coef=ENT, action_space=sp, nvec=([2, 4] if space == "multi_binary" else NVEC) if sp == "multi_discrete" else None)
        with pytest.raises(core_mod.PPOError, match=r"\[-1\].*action space"):
            c.load_meta_txt(other)
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode,uniform", [("md", 0.5 * (0.25 + 1.0 / 3.0)), ("mb", 0.5)])
def test_cli_bandit_train_save_load_eval(tmp_path, mode, uniform):
    host = os.path.join(ROOT, "ppo_cpp_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    exe = os.path.join(host, "bin", "ppo_cpp")
    common = ["--env", f"bandit_{mode}", "--threads", "4", "--seed", "5"]
    r = subprocess.run([exe, "-d", str(tmp_path / "exp"), "--id", "m0", "--hidden", "64,64", "--steps", "65536", "--lr", "3e-3",
                        "--num_epochs", "4", "--batch_steps", "512", "--saves", "1", *common], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    ck = tmp_path / "exp" / "checkpoints" / "m0"
    side = [f for f in os.listdir(ck) if f.endswith(".json")]
    space = "multi_discrete" if mode == "md" else "multi_binary"
    text = open(ck / side[0]).read()
    assert f'"{space}"' in text and (('"nvec"' in text) == (mode == "md")), text
    prefix = str(ck / side[0][:-len(".json")])
    A = 7 if mode == "md" else 4
    assert os.path.getsize(prefix + ".data-00000-of-00001") == 4 * mg.param_layout(4, A, 64, 64, action_space=space)["__total__"][0]
    # learning: the mean reward per step of the last updates, from the rollout's episode rewards (16-step episodes)
    rows = [l for l in open(tmp_path / "exp" / "tensorboard" / "m0" / "episode_reward.csv").read().split("\n")[1:] if l]
    ep = np.array([float(l.split(",")[1]) for l in rows])
    assert ep[-32:].mean() / 16.0 > uniform + 0.1, (ep[:8].mean() / 16.0, ep[-32:].mean() / 16.0)
    r = subprocess.run([exe, "-p", prefix, "--duration", "0.3", *common], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "episode_reward" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    r = subprocess.run([exe, "-p", prefix, "--duration", "0.3", "--env", "bandit", "--seed", "5"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0  # a checkpoint of another action space is refused


# ------------------------------------------------------------------ sharded updates (tests/mgpu_multi_action_worker.py)
WORLDS = (1, 2)
MGPU_TIMEOUT = 1200
_MGPU_RUNS = {}


def _free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _mgpu_launch(world, out_dir):
    import signal
    import sys
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "torch.distributed.run", "--nnodes", "1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
        "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "mgpu_multi_action_worker.py"), str(out_dir)]
    # its own session: on a timeout the whole process group goes, so no rank is left running
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, start_new_session=True)
    try:
        log, _ = p.communicate(timeout=MGPU_TIMEOUT)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        log, _ = p.communicate()
        return False, f"timed out after {MGPU_TIMEOUT} s\n{log[-6000:]}"
    return p.returncode == 0, log[-6000:]


@pytest.fixture(scope="module")
def mgpu_runs(tmp_path_factory):
    """mgpu_runs(W) -> the worker's output directory of world size W (launched on first use, once per module)."""
    def get(world):
        if torch.cuda.device_count() < world:
            pytest.skip(f"needs {world} GPUs, the box has {torch.cuda.device_count()}")
        if world not in _MGPU_RUNS:
            out = tmp_path_factory.mktemp(f"mgpu_multi_action_w{world}")
            _MGPU_RUNS[world] = (out,) + _mgpu_launch(world, out)
        out, ok, log = _MGPU_RUNS[world]
        assert ok, f"world {world}: the worker failed\n{log}"
        return out
    return get


def _mgpu_cases():
    import mgpu_multi_action_worker as w
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", ["md_fused", "md_tile", "md_nccl", "mb_fused", "mb_tile", "mb_nccl"])
def test_sharded_update_vs_fp64_learner(mgpu_runs, name, world):
    """A sharded update against the single-GPU fp64 learner on the global rollout (every rank's rows, rank r holding global
    envs [r * n_envs, (r + 1) * n_envs)), with the permutations the cores report and the Adam state carried over two annealed
    updates: every rank's params and Adam state bit-identical to rank 0's, params and Adam moments against the learner, and all
    five losses — the entropy among them, whose per-sample column is scaled by the rank count and divided by it again after the
    reduce.  World 1 runs the same cases on one GPU (no exchange), which checks the harness and the reference on any box."""
    w = _mgpu_cases()
    assert (w.O, w.NVEC, w.NB) == (O, NVEC, NB)
    spec = w.CASES[name]
    if world == 1 and spec.get("p2p") is False:
        pytest.skip("the NCCL fallback exchanges between two or more ranks")
    out = mgpu_runs(world)
    ranks = [dict(np.load(os.path.join(out, f"{name}_r{r}.npz"))) for r in range(world)]
    r0 = ranks[0]
    what = f"{name} at world {world}"
    space = w.HEADS[spec["head"]]["action_space"]
    fam = str(r0["family_train"])
    assert ("train_tile_kernel" if "PPO_DISABLE_FUSED" in spec.get("env", ()) else "train_fused_kernel") in fam, (what, fam)
    for r, d in enumerate(ranks):
        assert not bool(d["comm_error"]), f"{what}: a peer-mailbox wait timed out on rank {r}"
        for t in ("params", "adam_m", "adam_v", "beta1_power", "beta2_power"):
            assert np.array_equal(d[t], r0[t]), f"{what}: rank {r} {t} differs from rank 0's"
    ent, vf, clip, b1, b2, eps = r0["hparams"].astype(np.float64)
    h1, h2 = spec["hidden"]
    lay, P, _ = layout(space, h1, h2)
    loss = partial(loss_grad_ref, activation=spec.get("activation", "tanh"), space=space, h1=h1, h2=h2, ent_coef=ent, vf_coef=vf)
    p0 = r0["p0"]
    p, state = p0, {}
    for u in range(spec["updates"]):
        bufs = {b: np.concatenate([d[f"u{u}_{b}"] for d in ranks], axis=0) for b in ("obs", "actions", "returns", "values", "neglogpacs")}
        perms = r0[f"u{u}_perms"]
        for r, d in enumerate(ranks):
            assert np.array_equal(d[f"u{u}_perms"], perms), f"{what}: rank {r} trained on other permutations"
        lr, cr = (float(x) for x in r0[f"u{u}_schedule"])
        p, want = learner_ref(p, bufs, perms, spec["nmb"], lr, cr, loss, clip=clip, b1=b1, b2=b2, eps=eps, state=state)
        got = r0[f"u{u}_losses"]
        assert np.allclose(got, want, rtol=2e-5, atol=1e-6), (what, f"update {u} losses", got, want)
    got = r0["params"]
    moved = np.abs(p[:P] - p0[:P]).max()
    diff = np.abs(got[:P] - p[:P]).max()
    assert diff < max(5e-4, 4e-5 * spec["epochs"] * spec["nmb"]) * moved, (what, "params", diff / moved)
    assert np.array_equal(got[P:], p0[P:])
    for key in ("adam_m", "adam_v"):
        for off, s in lay:
            sl = slice(off, off + int(np.prod(s)))
            assert rel_err(r0[key][sl], state[key[-1]][sl]) < 2e-4, (what, key, off, rel_err(r0[key][sl], state[key[-1]][sl]))
    assert float(r0["beta1_power"][0]) == pytest.approx(state["b1p"], rel=1e-5)
    assert float(r0["beta2_power"][0]) == pytest.approx(state["b2p"], rel=1e-5)
