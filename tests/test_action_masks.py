"""Invalid-action masks on Discrete and MultiDiscrete heads (sb3-contrib's MaskableCategorical, ppo_core_set_action_masking).

The reference is an fp64 PyTorch autograd restatement of the PPO2 loss as sb3-contrib writes the masked head: forbidden logits
replaced by -1e8 (torch.where, so no gradient reaches them), log_softmax for neglogp, and the entropy as -sum where(mask, p log p, 0).
GPU tests (the F and T families, tanh and ReLU): masked policy steps with given uniforms, deterministic actions, loss and gradients,
whole updates against the fp64 learner of test_vf_clip_and_schedules (the masks ride along with the actions through a wrapper loss),
bit-identity with the unmasked core when every action is allowed, the host-env protocol and every error rule.  CPU test: the masked
bandit env of the CLI."""
import os
import subprocess
from functools import partial

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_err
from ppo_cpp_b200 import meta_graph as mg
from test_vf_clip_and_schedules import _tf_clip, _tf_max, learner_ref, value_loss

TOL = 1e-5
ENT = 0.01
O = 6
N_DISC = 7
NVEC = [3, 5, 2]  # slices that straddle the Philox blocks of 4, a tail of 2
SPACES = {"discrete": dict(act_dim=N_DISC), "multi_discrete": dict(nvec=NVEC)}
FT = [((), "fused"), (("PPO_DISABLE_FUSED",), "tile")]


def width(space):
    return N_DISC if space == "discrete" else sum(NVEC)


def slices(space):
    if space == "discrete":
        return [(0, N_DISC)]
    off = np.concatenate([[0], np.cumsum(NVEC)])
    return [(int(off[i]), int(off[i + 1])) for i in range(len(NVEC))]


# ------------------------------------------------------------------ layout, masks and the fp64 reference
def layout(space, h1, h2):
    lay = mg.param_layout(O, width(space), h1, h2, action_space=space)
    order = [t for t in mg.TENSOR_ORDER[:mg.N_TRAINABLE_TENSORS] if t != mg.LOGSTD]
    return [lay[t] for t in order], lay["model/q/w"][0], lay["__total__"][0]


def rand_params(rng, space, h1, h2):
    _, _, Pq = layout(space, h1, h2)
    p = (rng.standard_normal(Pq) * min(0.3, 1.5 / np.sqrt(max(h1, h2)))).astype(np.float32)
    off = mg.param_layout(O, width(space), h1, h2, action_space=space)["model/pi/w"][0]
    p[off:off + h2 * width(space)] *= 4.0
    return p


def forward_ref(params, obs, activation, space, h1, h2):
    lay, _, _ = layout(space, h1, h2)
    t = [params.astype(np.float64)[off:off + int(np.prod(s))].reshape(s) for off, s in lay]
    f = np.tanh if activation == "tanh" else (lambda z: np.maximum(z, 0.0))
    x = obs.astype(np.float64)
    logits = f(f(x @ t[0] + t[1]) @ t[4] + t[5]) @ t[10] + t[11]
    v = (f(f(x @ t[2] + t[3]) @ t[6] + t[7]) @ t[8] + t[9])[:, 0]
    return logits, v


def rand_masks(rng, space, B, p=0.5):
    """Random 0 / 1 masks [B, A] with about p of the logits allowed and at least one per slice; every 7th row allows a single logit
    per slice, every 5th row everything."""
    m = (rng.uniform(size=(B, width(space))) < p).astype(np.uint8)
    for i, (a, b) in enumerate(slices(space)):
        empty = m[:, a:b].sum(1) == 0
        m[empty, a + rng.integers(0, b - a, int(empty.sum()))] = 1
        m[::7, a:b] = 0
        m[np.arange(0, B, 7), a + (np.arange(0, B, 7) + i) % (b - a)] = 1
    m[::5] = 1
    return m


def masked_nlp_ent(logits, act, mask, space):
    """sb3-contrib's MaskableCategorical per slice, summed: -1e8 in the forbidden logits, neglogp of act and the entropy
    -sum where(mask, p log p, 0); torch fp64."""
    nlp, ent = 0.0, 0.0
    for i, (a, b) in enumerate(slices(space)):
        mk = mask[:, a:b]
        li = torch.where(mk, logits[:, a:b], torch.full_like(logits[:, a:b], -1e8))
        lp = torch.log_softmax(li, 1)
        nlp = nlp - lp.gather(1, act[:, i:i + 1].long())[:, 0]
        ent = ent - torch.where(mk, torch.exp(lp) * lp, torch.zeros_like(lp)).sum(1)
    return nlp, ent


def neglogp_np(logits, act, mask, space):
    n, _ = masked_nlp_ent(torch.tensor(logits), torch.tensor(np.asarray(act, np.float64)), torch.tensor(mask.astype(bool)), space)
    return n.numpy()


def loss_grad_ref(params, obs, act, adv, ret, old_nlp, old_v, cr, activation, space, h1, h2, masks=None, ent_coef=ENT, vf_coef=0.5,
                  vf="shared", cr_vf=0.0):
    lay, P, _ = layout(space, h1, h2)
    p = torch.tensor(np.asarray(params[:P], np.float64), requires_grad=True)
    pi0w, pi0b, vf0w, vf0b, pi1w, pi1b, vf1w, vf1b, vfw, vfb, piw, pib = [p[off:off + int(np.prod(s))].reshape(s) for off, s in lay]
    f = torch.tanh if activation == "tanh" else torch.relu
    x = torch.tensor(np.asarray(obs, np.float64))
    a = torch.tensor(np.asarray(act, np.float64))
    mk = torch.tensor(np.asarray(masks) > 0.5)
    adv, R, onl, ov = (torch.tensor(np.asarray(z, np.float64).ravel()) for z in (adv, ret, old_nlp, old_v))
    logits = f(f(x @ pi0w + pi0b) @ pi1w + pi1b) @ piw + pib
    v = (f(f(x @ vf0w + vf0b) @ vf1w + vf1b) @ vfw + vfb)[:, 0]
    nlp, ent = masked_nlp_ent(logits, a, mk, space)
    ratio = torch.exp(onl - nlp)
    pg = _tf_max(-adv * ratio, -adv * _tf_clip(ratio, torch.tensor(1.0 - cr, dtype=torch.float64), torch.tensor(1.0 + cr, dtype=torch.float64))).mean()
    vfl = 0.5 * value_loss(v, ov, R, vf, cr, cr_vf).mean()
    ent = ent.mean()
    loss = pg - ent * ent_coef + vfl * vf_coef
    loss.backward()
    with torch.no_grad():
        kl = 0.5 * ((nlp - onl) ** 2).mean()
        cf = ((ratio - 1.0).abs() > cr).double().mean()
    return p.grad.numpy().copy(), np.array([pg.item(), vfl.item(), ent.item(), kl.item(), cf.item()])


def learner_loss(params, obs, act_and_mask, *rest, space, **kw):
    """learner_ref's loss: the minibatch's actions with their masks behind them in the same rows (rollout_get("actions") | "action_masks")."""
    k = len(slices(space))
    return loss_grad_ref(params, obs, act_and_mask[:, :k], *rest, space=space, masks=act_and_mask[:, k:], **kw)


def masked_gumbel(logits, u, mask, space):
    with np.errstate(divide="ignore"):
        g = np.where(mask > 0, logits - np.log(-np.log(u.astype(np.float64))), -np.inf)
    return np.stack([np.argmax(g[:, a:b], 1) for a, b in slices(space)], 1).astype(np.float32), g


def uniform_fixture(rng, logits, mask, space):
    """Uniforms whose masked Gumbel-max fp32 rounding cannot change: in every slice the maximum over the allowed logits is at least
    1e-3 above the runner-up.  Returns (u, the actions they give)."""
    u = rng.uniform(0.0, 1.0, logits.shape)
    for a, b in slices(space):
        for _ in range(200):
            _, g = masked_gumbel(logits, u, mask, space)
            srt = np.sort(g[:, a:b], 1)
            bad = (srt[:, -1] - srt[:, -2] < 1e-3) & np.isfinite(srt[:, -2])
            if not bad.any():
                break
            u[bad, a:b] = rng.uniform(0.0, 1.0, (int(bad.sum()), b - a))
    return u.astype(np.float32), masked_gumbel(logits, u, mask, space)[0]


def allowed(acts, mask, space):
    """Every action column's index allowed by its row's mask."""
    return all(np.all(mask[np.arange(len(acts)), a + acts[:, i].astype(int)] == 1) for i, (a, b) in enumerate(slices(space)))


def sample_masked(rng, logits, mask, space):
    cols = []
    for a, b in slices(space):
        q = np.where(mask[:, a:b] > 0, np.exp(logits[:, a:b] - logits[:, a:b].max(1, keepdims=True)), 0.0)
        q /= q.sum(1, keepdims=True)
        cols.append([rng.choice(b - a, p=r) for r in q])
    return np.array(cols, np.float32).T


# ------------------------------------------------------------------ CPU: the masked bandit env of the CLI
def test_host_bandit_mask_env(tmp_path):
    """bandit_mask: a Discrete(4) contextual bandit whose context forbids one or two actions, never the rewarded one; it counts the
    illegal actions it receives.  A perfect policy earns 1 per step, a legal wrong one 0, and only an illegal action counts."""
    src = tmp_path / "b.cpp"
    src.write_text('#include "env_bandit.hpp"\n#include <cstdio>\nint main() {\n'
                   '  BanditEnv e(4, 0, 3, BanditEnv::MASKED);\n  Mat obs = e.reset();\n'
                   '  int ok = e.get_action_space() == Env::SPACE_DISCRETE() && e.get_action_space_size() == 4 && e.has_action_mask();\n'
                   '  float good = 0, wrong = 0; int bad_masks = 0, seen = 0, forb = 0;\n'
                   '  for (int t = 0; t < 96; ++t) {\n'
                   '    Mat m = e.get_action_mask();\n    int c = 0, n_allowed = 0;\n'
                   '    for (int k = 0; k < 4; ++k) { if (obs(0, k) > 0.5f) c = k; n_allowed += m(0, k) > 0.5f; }\n'
                   '    seen |= 1 << c;\n    if (m(0, (c + 1) % 4) < 0.5f || n_allowed < 2 || n_allowed > 3) ++bad_masks;\n'
                   '    int a = (c + 1) % 4;\n    if (t % 3 == 1) { a = (c + 2) % 4; while (m(0, a) < 0.5f || a == (c + 1) % 4) a = (a + 1) % 4; }\n'
                   '    if (t % 3 == 2) { a = 0; while (m(0, a) > 0.5f) ++a; ++forb; }\n'
                   '    Mat act(1, 1); act(0, 0) = (float)a;\n    auto r = e.step(act);\n'
                   '    if (t % 3 == 0) good += r[1](0, 0); else if (t % 3 == 1) wrong += r[1](0, 0);\n    obs = r[0];\n  }\n'
                   '  std::printf("%d %g %g %d %d %ld %d\\n", ok, good, wrong, bad_masks, __builtin_popcount(seen), e.illegal_actions(), forb);\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "b"
    subprocess.run(["g++", "-std=c++14", "-O1", "-I", os.path.join(ROOT, "ppo_cpp_b200", "host"), "-o", str(exe), str(src)], check=True)
    ok, good, wrong, bad_masks, seen, illegal, forb = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert (int(ok), float(good), float(wrong), int(bad_masks), int(seen)) == (1, 32.0, 0.0, 0, 4)
    assert int(illegal) == int(forb) == 32


# ------------------------------------------------------------------ GPU
def _core(core_mod, monkeypatch, space, env=(), masking=True, **kw):
    for e in env:
        monkeypatch.setenv(e, "1")
    kw.setdefault("obs_dim", O)
    kw = {**SPACES[space], **kw}
    c = core_mod.PPOCore(action_space=space, **kw)
    for e in env:
        monkeypatch.delenv(e)
    assert not c.action_masking  # off at creation
    c.action_masking = masking
    assert c.action_masking == masking
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ["tanh", "relu"])
@pytest.mark.parametrize("env,fam", FT)
@pytest.mark.parametrize("space", sorted(SPACES))
def test_policy_step_masked_vs_fp64(monkeypatch, space, env, fam, activation):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(3)
    B = 3000
    p = rand_params(rng, space, 64, 64)
    obs = rng.standard_normal((B, O)).astype(np.float32)
    logits, v64 = forward_ref(p, obs, activation, space, 64, 64)
    mask = rand_masks(rng, space, B)
    u, want = uniform_fixture(rng, logits, mask, space)
    c = _core(core_mod, monkeypatch, space, env, activation=activation, hidden1=64, hidden2=64, n_envs=B, n_steps=2, nminibatches=1)
    assert fam in c.kernel_family("policy") and fam in c.kernel_family("train")
    c.set_tensor("params", p)
    a, v, nlp = c.policy_step(obs, u, mask=mask)
    assert allowed(a, mask, space)
    assert np.array_equal(a, want)
    assert rel_err(nlp, neglogp_np(logits, want, mask, space)) < TOL
    _, v_plain, _ = c.policy_step(obs, u)
    assert np.array_equal(v, v_plain) and rel_err(v, v64) < TOL  # the value tower does not see the mask
    # deterministic action: the masked argmax (rows whose allowed top two are apart)
    det = c.policy_mean(obs, mask=mask)
    assert allowed(det, mask, space)
    ml = np.where(mask > 0, logits, -np.inf)
    sep = np.ones(B, bool)
    for a_, b_ in slices(space):
        srt = np.sort(ml[:, a_:b_], 1)
        sep &= (srt[:, -1] - srt[:, -2] > 1e-4) | ~np.isfinite(srt[:, -2])
    want_det = np.stack([np.argmax(ml[:, a_:b_], 1) for a_, b_ in slices(space)], 1).astype(np.float32)
    assert sep.mean() > 0.9 and np.array_equal(det[sep], want_det[sep])
    # Philox noise: never a forbidden action, over several draws
    for _ in range(3):
        a, _, nlp = c.policy_step(obs, mask=mask)
        assert allowed(a, mask, space) and rel_err(nlp, neglogp_np(logits, a, mask, space)) < TOL
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ["tanh", "relu"])
@pytest.mark.parametrize("space", sorted(SPACES))
def test_loss_grad_masked_vs_fp64(monkeypatch, space, activation):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(5)
    h, B = 64, 1000
    p = rand_params(rng, space, h, h)
    obs = rng.standard_normal((B, O)).astype(np.float32)
    logits, v = forward_ref(p, obs, activation, space, h, h)
    mask = rand_masks(rng, space, B)
    dead = slices(space)[-1][0] + 1  # a logit forbidden in every row
    mask[:, dead] = 0
    for a_, b_ in slices(space):  # keep every slice non-empty
        empty = mask[:, a_:b_].sum(1) == 0
        mask[empty, a_] = 1
    act = sample_masked(rng, logits, mask, space)
    old_nlp = (neglogp_np(logits, act, mask, space) + 0.1 * rng.standard_normal(B)).astype(np.float32)
    old_v = (v + 0.3 * rng.standard_normal(B)).astype(np.float32)
    ret = (v + 0.3 + 0.5 * rng.standard_normal(B)).astype(np.float32)
    adv = rng.standard_normal(B).astype(np.float32)
    data = (obs, act, adv, ret, old_nlp, old_v)
    lay, P, _ = layout(space, h, h)
    piw, pib = lay[10], lay[11]
    A = width(space)
    for vf, cr_vf in (("shared", None), ("separate", 0.15)):
        g64, l64 = loss_grad_ref(p, *data, 0.2, activation, space, h, h, masks=mask, vf=vf, cr_vf=cr_vf or 0.0)
        outs = []
        for env, fam in FT:
            c = _core(core_mod, monkeypatch, space, env, activation=activation, hidden1=h, hidden2=h, n_envs=4, n_steps=8, nminibatches=4, ent_coef=ENT)
            assert fam in c.kernel_family("train")
            c.vf_clip = vf
            c.set_tensor("params", p)
            g, l = c.loss_grad(*data, 0.2, cliprange_vf=cr_vf, masks=mask)
            c.close()
            for t, (off, s) in enumerate(lay):
                sl = slice(off, off + int(np.prod(s)))
                assert rel_err(g[sl], g64[sl]) < TOL, (vf, fam, t, rel_err(g[sl], g64[sl]))
            for k in range(5):
                assert np.isclose(l[k], l64[k], rtol=TOL, atol=1e-7), (vf, fam, k, l, l64)
            assert g[pib[0] + dead] == 0.0 and np.all(g[piw[0]:piw[0] + h * A].reshape(h, A)[:, dead] == 0.0)
            outs.append(g)
        assert rel_err(outs[0], outs[1]) < 2e-6
    # the mask matters: without it the gradient differs
    g_open, _ = loss_grad_ref(p, *data, 0.2, activation, space, h, h, masks=np.ones_like(mask))
    assert rel_err(g_open, g64) > 1e-3


def _masked_rollout(c, rng, space, n_envs, n_steps, obs0, mask0, masks=None):
    """The host-env protocol with random observations and masks; returns (actions [T, N, k], the masks in force at each step [T, N, A],
    the last mask)."""
    if obs0 is not None:
        c.runner_reset(obs0, mask=mask0)
    acts, used = [], []
    cur = mask0
    for t in range(n_steps):
        acts.append(c.runner_act(t).copy())
        used.append(cur)
        cur = rand_masks(rng, space, n_envs) if masks is None else masks[t]
        c.runner_observe(t, rng.standard_normal((n_envs, O)).astype(np.float32), rng.standard_normal(n_envs).astype(np.float32),
                         (rng.uniform(size=n_envs) < 0.05).astype(np.float32), mask=cur)
    c.runner_finish()
    return np.stack(acts), np.stack(used), cur


@pytest.mark.gpu
@pytest.mark.parametrize("env,fam", FT)
@pytest.mark.parametrize("space", sorted(SPACES))
def test_host_env_protocol_stores_and_carries_masks(monkeypatch, space, env, fam):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(8)
    n_envs, n_steps = 96, 12
    c = _core(core_mod, monkeypatch, space, env, hidden1=64, hidden2=64, n_envs=n_envs, n_steps=n_steps, nminibatches=4, seed=31)
    c.set_tensor("params", rand_params(rng, space, 64, 64))
    acts, used, last = _masked_rollout(c, rng, space, n_envs, n_steps, rng.standard_normal((n_envs, O)).astype(np.float32),
                                       rand_masks(rng, space, n_envs))
    for t in range(n_steps):
        assert allowed(acts[t], used[t], space), t
    got = c.rollout_get("action_masks")
    assert got.shape == (n_envs * n_steps, width(space)) and got.dtype == np.float32
    assert np.array_equal(got.reshape(n_envs, n_steps, -1), used.transpose(1, 0, 2).astype(np.float32))  # flat row = env * n_steps + t
    assert np.array_equal(c.rollout_get("actions").reshape(n_envs, n_steps, -1), acts.transpose(1, 0, 2))
    # the next rollout's step 0 uses the mask of the last observe, as it uses its observation
    a0 = c.runner_act(0)
    assert allowed(a0, last, space)
    assert np.array_equal(c.rollout_get("action_masks").reshape(n_envs, n_steps, -1)[:, 0], last.astype(np.float32))
    # plain calls allow everything: observe without a mask
    c.runner_observe(0, rng.standard_normal((n_envs, O)).astype(np.float32), np.zeros(n_envs, np.float32), np.zeros(n_envs, np.float32))
    c.runner_act(1)
    assert np.all(c.rollout_get("action_masks").reshape(n_envs, n_steps, -1)[:, 1] == 1.0)
    c.close()


def _three_cores(core_mod, monkeypatch, space, env, **kw):
    return [_core(core_mod, monkeypatch, space, env, masking=m, **kw) for m in (False, True, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("env,fam", FT)
@pytest.mark.parametrize("space", sorted(SPACES))
def test_all_allowed_is_bit_identical_to_unmasked(monkeypatch, space, env, fam):
    """An unmasked core, a masking core fed all-ones masks, and a masking core driven through the plain entry points: actions,
    neglogp, rollout buffers, parameters, Adam state and losses over two updates are bit-identical."""
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(17)
    n_envs, n_steps, h = 128, 16, 64
    kw = dict(hidden1=h, hidden2=h, n_envs=n_envs, n_steps=n_steps, nminibatches=4, noptepochs=2, ent_coef=ENT, seed=5)
    p = rand_params(rng, space, h, h)
    obs0 = rng.standard_normal((n_envs, O)).astype(np.float32)
    traj = [(rng.standard_normal((n_envs, O)).astype(np.float32), rng.standard_normal(n_envs).astype(np.float32),
             (rng.uniform(size=n_envs) < 0.05).astype(np.float32)) for _ in range(2 * n_steps)]
    ones = np.ones((n_envs, width(space)), np.uint8)
    res = []
    for i, c in enumerate(_three_cores(core_mod, monkeypatch, space, env, **kw)):
        mk = ones if i == 1 else None
        c.set_tensor("params", p)
        out = [c.policy_step(obs0, mask=mk), c.policy_mean(obs0, mask=mk)]
        c.runner_reset(obs0, mask=mk)
        c.shuffle_seed(3)
        for u in range(2):
            for t in range(n_steps):
                out.append(c.runner_act(t).copy())
                c.runner_observe(t, *traj[u * n_steps + t], mask=mk)
            c.runner_finish()
            out += [c.rollout_get(n) for n in ("obs", "actions", "values", "neglogpacs", "returns", "dones")]
            out.append(c.train_update(3e-4, 0.2))
        out += [c.get_tensor(n) for n in ("params", "adam_m", "adam_v", "beta1_power", "beta2_power")]
        if i:
            assert np.all(c.rollout_get("action_masks") == 1.0)
        res.append(out)
        c.close()
    for k in range(len(res[0])):
        flat = [np.concatenate([np.ravel(q) for q in r[k]]) if isinstance(r[k], tuple) else np.ravel(r[k]) for r in res]
        assert np.array_equal(flat[0], flat[1]) and np.array_equal(flat[0], flat[2]), k


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ["tanh", "relu"])
@pytest.mark.parametrize("env,fam", FT)
@pytest.mark.parametrize("shuffle", ["device", "host"])
@pytest.mark.parametrize("space", sorted(SPACES))
def test_train_update_masked_vs_fp64_learner(monkeypatch, space, shuffle, env, fam, activation):
    """Three annealed updates on a masking core against the fp64 learner (Adam state carried), with CUDA graphs (replayed, not rebuilt,
    after the first update) and without them (bit-identical)."""
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(21)
    h, n_envs, n_steps, nmb, epochs = 64, 128, 16, 4, 2
    flat = rand_params(rng, space, h, h)
    obs0 = rng.standard_normal((n_envs, O)).astype(np.float32)
    mask0 = rand_masks(rng, space, n_envs)
    masks = [rand_masks(rng, space, n_envs) for _ in range(3 * n_steps)]
    sw = ("PPO_DISABLE_GPU_SHUFFLE",) if shuffle == "host" else ()
    runs = []
    for graph in (True, False):
        c = _core(core_mod, monkeypatch, space, env + sw + (() if graph else ("PPO_DISABLE_GRAPH",)), activation=activation, hidden1=h,
                  hidden2=h, n_envs=n_envs, n_steps=n_steps, nminibatches=nmb, noptepochs=epochs, ent_coef=ENT, seed=9)
        assert fam in c.kernel_family("train")
        c.set_tensor("params", flat)
        c.shuffle_seed(42)
        r = np.random.default_rng(77)
        out, builds = [], []
        for u in range(3):
            acts, used, _ = _masked_rollout(c, r, space, n_envs, n_steps, obs0 if u == 0 else None, mask0, masks[u * n_steps:(u + 1) * n_steps])
            bufs = {n: c.rollout_get(n) for n in ("obs", "actions", "returns", "values", "neglogpacs")}
            bufs["actions"] = np.concatenate([bufs["actions"], c.rollout_get("action_masks")], 1)
            lr, cr = 3.9e-4 * (1.0 - u / 3), 0.2 - 0.05 * u
            losses = c.train_update(lr, cr)
            out.append((bufs, [c.train_get_permutation(e) for e in range(epochs)], lr, cr, losses))
            builds.append(c.graph_builds())
        out.append(tuple(c.get_tensor(n) for n in ("params", "adam_m", "adam_v")))
        if graph:
            assert builds[0] > 0 and builds[1] == builds[0] and builds[2] == builds[0], builds
        else:
            assert builds[-1] == 0
        runs.append(out)
        c.close()
    for x, y in zip(runs[0][-1], runs[1][-1]):
        assert np.array_equal(x, y)  # graphs and eager launches: bit-identical
    for u in range(3):
        assert np.array_equal(runs[0][u][4], runs[1][u][4])
    p, state = flat, {}
    loss = partial(learner_loss, activation=activation, space=space, h1=h, h2=h)
    _, P, _ = layout(space, h, h)
    for bufs, perms, lr, cr, losses in runs[0][:3]:
        p, want = learner_ref(p, bufs, perms, nmb, lr, cr, loss, state=state)
        assert np.allclose(losses, want, rtol=2e-5, atol=1e-6), (losses, want)
    got = runs[0][-1][0]
    moved = np.abs(p[:P] - flat[:P]).max()
    assert np.abs(got[:P] - p[:P]).max() < max(5e-4, 4e-5 * 3 * epochs * nmb) * moved


def _lib_call(c, fn, *args):
    return getattr(c.lib, fn)(c._h, *args)


@pytest.mark.gpu
@pytest.mark.parametrize("space", sorted(SPACES))
def test_error_rules(monkeypatch, space):
    from ppo_cpp_b200 import core as core_mod
    from ppo_cpp_b200 import _lib
    rng = np.random.default_rng(4)
    n_envs, n_steps, A = 16, 4, width(space)
    c = _core(core_mod, monkeypatch, space, hidden1=64, hidden2=64, n_envs=n_envs, n_steps=n_steps, nminibatches=2, masking=False)
    obs = rng.standard_normal((n_envs, O)).astype(np.float32)
    good = rand_masks(rng, space, n_envs)
    # _masked calls with masking off
    k0 = np.zeros((n_envs, len(slices(space))), np.float32)
    z = np.zeros(n_envs, np.float32)
    for fn in (lambda: c.policy_step(obs, mask=good), lambda: c.policy_mean(obs, mask=good), lambda: c.runner_reset(obs, mask=good),
               lambda: c.runner_observe(0, obs, z, z, mask=good), lambda: c.loss_grad(obs, k0, z, z, z, z, 0.2, masks=good),
               lambda: c.rollout_get("action_masks"), lambda: c.rollout_set("action_masks", np.ones((n_envs * n_steps, A), np.float32))):
        with pytest.raises(core_mod.PPOError, match=r"\[-1\].*masking is off"):
            fn()
    c.action_masking = True
    # the Python mirror refuses what the library cannot tell apart: another shape (it would read past the array) and non-integers
    for m in (good[:, :A - 1], good[:-1], good.ravel(), np.where(good > 0, 0.5, 0.0)):
        with pytest.raises(ValueError, match="action mask"):
            c.policy_step(obs, mask=m)
    # a value other than 0 / 1, naming row and column
    bad = good.copy()
    bad[5, 2] = 2
    with pytest.raises(core_mod.PPOError, match=r"\[-1\].*row 5, column 2 is 2"):
        c.policy_step(obs, mask=bad)
    # a categorical with no allowed logit, naming row (and slice)
    a_, b_ = slices(space)[-1]
    bad = good.copy()
    bad[3, a_:b_] = 0
    want = r"row 3 allows no action" if space == "discrete" else rf"row 3, slice {len(NVEC) - 1} \(logits {a_} \.\. {b_ - 1}\)"
    for fn in (lambda: c.policy_step(obs, mask=bad), lambda: c.runner_reset(obs, mask=bad),
               lambda: c.runner_observe(0, obs, np.zeros(n_envs), np.zeros(n_envs), mask=bad)):
        with pytest.raises(core_mod.PPOError, match=r"\[-1\].*" + want):
            fn()
    # a recorded action its mask forbids: rollout_set and loss_grad_masked
    c.set_tensor("params", rand_params(rng, space, 64, 64))
    c.runner_reset(obs, mask=good)
    for t in range(n_steps):
        c.runner_act(t)
        c.runner_observe(t, obs, np.zeros(n_envs), np.zeros(n_envs), mask=good)
    c.runner_finish()
    acts, masks = c.rollout_get("actions"), c.rollout_get("action_masks")
    row, col = 6, len(slices(space)) - 1
    lo, hi = slices(space)[col]
    k = int(acts[row, col])
    forb = masks.copy()
    forb[row, lo:hi] = 0
    forb[row, lo + (k + 1) % (hi - lo)] = 1  # the slice allows one other index
    with pytest.raises(core_mod.PPOError, match=rf"\[-1\].*row {row}, column {col}: action {k} is forbidden"):
        c.rollout_set("action_masks", forb)
    zeros = np.zeros(len(acts), np.float32)
    with pytest.raises(core_mod.PPOError, match=rf"\[-1\].*row {row}, column {col}: action {k} is forbidden"):
        c.loss_grad(c.rollout_get("obs"), acts, zeros, zeros, zeros, zeros, 0.2, masks=forb.astype(np.uint8))
    c.rollout_set("action_masks", masks)  # the recorded masks go back in
    assert np.array_equal(c.rollout_get("action_masks"), masks)
    c.rollout_set("actions", acts)  # setting actions allows everything in those rows
    assert np.all(c.rollout_get("action_masks") == 1.0)
    # rollout_host / replay take no masks
    for fn in (lambda: c.runner_rollout_replay(np.zeros((n_steps, n_envs, O)), np.zeros((n_steps, n_envs)), np.zeros((n_steps, n_envs))),
               lambda: c.runner_rollout_host(lambda t, a: (obs, np.zeros(n_envs), np.zeros(n_envs)))):
        with pytest.raises(core_mod.PPOError, match=r"\[-4\]"):
            fn()
    # a device-memory mask with an empty slice: reported by the next finish, update, minibatch step and sync
    dev_obs = torch.tensor(obs, device="cuda")
    dev_bad = torch.tensor(bad, device="cuda")
    dev_act = torch.zeros((n_envs, len(slices(space))), device="cuda")
    c.train_set_permutation(np.arange(n_envs * n_steps))
    for check in ("finish", "update", "minibatch", "sync"):
        assert _lib_call(c, "ppo_runner_reset_masked", dev_obs.data_ptr(), dev_bad.data_ptr(), _lib.PPO_DEVICE) == 0
        if check == "minibatch":
            with pytest.raises(core_mod.PPOError, match=r"\[-1\].*device-memory action mask: mask row 3"):
                c.train_minibatch(0, 3e-4, 0.2)
        elif check == "finish":
            for t in range(n_steps):
                c.runner_act(t)
                c.runner_observe(t, obs, np.zeros(n_envs), np.zeros(n_envs), mask=good)
            with pytest.raises(core_mod.PPOError, match=r"\[-1\].*device-memory action mask: mask row 3"):
                c.runner_finish()
        elif check == "update":
            with pytest.raises(core_mod.PPOError, match=r"\[-1\].*device-memory action mask: mask row 3"):
                c.train_update(3e-4, 0.2)
        else:
            assert _lib_call(c, "ppo_policy_step_masked", dev_obs.data_ptr(), n_envs, None, dev_bad.data_ptr(), dev_act.data_ptr(), None, None,
                             _lib.PPO_DEVICE) == 0
            torch.cuda.synchronize()
            assert allowed(dev_act.cpu().numpy(), np.ones_like(bad), space)
            with pytest.raises(core_mod.PPOError, match=r"\[-1\].*device-memory action mask: mask row 3"):
                c.sync()
        c.sync()  # reported once
    # a device mask that is fine reports nothing
    assert _lib_call(c, "ppo_runner_reset_masked", dev_obs.data_ptr(), torch.tensor(good, device="cuda").data_ptr(), _lib.PPO_DEVICE) == 0
    c.sync()
    c.close()
    # Box and MultiBinary have no masks
    for sp, kw in (("box", dict(act_dim=4)), ("multi_binary", dict(act_dim=4))):
        d = core_mod.PPOCore(action_space=sp, obs_dim=O, n_envs=8, n_steps=4, nminibatches=2, **kw)
        with pytest.raises(core_mod.PPOError, match=r"\[-4\]"):
            d.action_masking = True
        assert not d.action_masking
        d.close()


@pytest.mark.gpu
def test_cli_bandit_mask_train_save_load_eval(tmp_path):
    """ppo2 --env bandit_mask: the policy never takes an illegal action, the reward rises above the uniform legal policy's, and a saved
    checkpoint evaluates with legal actions only."""
    host = os.path.join(ROOT, "ppo_cpp_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    exe = os.path.join(host, "bin", "ppo_cpp")
    common = ["--env", "bandit_mask", "--threads", "4", "--seed", "5"]
    r = subprocess.run([exe, "-d", str(tmp_path / "exp"), "--id", "m0", "--hidden", "64,64", "--steps", "65536", "--lr", "3e-3",
                        "--num_epochs", "4", "--batch_steps", "512", "--saves", "1", *common], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "illegal_actions 0" in r.stdout, r.stdout[-3000:]
    ck = tmp_path / "exp" / "checkpoints" / "m0"
    side = [f for f in os.listdir(ck) if f.endswith(".json")]
    prefix = str(ck / side[0][:-len(".json")])
    rows = [l for l in open(tmp_path / "exp" / "tensorboard" / "m0" / "episode_reward.csv").read().split("\n")[1:] if l]
    ep = np.array([float(l.split(",")[1]) for l in rows])
    uniform = 1.0 / 2.5  # one legal action of two or three is rewarded
    assert ep[-32:].mean() / 16.0 > uniform + 0.2 and ep[-32:].mean() > ep[:8].mean(), (ep[:8].mean() / 16.0, ep[-32:].mean() / 16.0)
    r = subprocess.run([exe, "-p", prefix, "--duration", "0.3", *common], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "episode_reward" in r.stdout and "illegal_actions 0" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


# ------------------------------------------------------------------ sharded masked updates (tests/mgpu_action_mask_worker.py)
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
        "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "mgpu_action_mask_worker.py"), str(out_dir)]
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
            out = tmp_path_factory.mktemp(f"mgpu_action_mask_w{world}")
            _MGPU_RUNS[world] = (out,) + _mgpu_launch(world, out)
        out, ok, log = _MGPU_RUNS[world]
        assert ok, f"world {world}: the worker failed\n{log}"
        return out
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", ["disc_fused", "disc_tile", "disc_nccl", "md_fused", "md_tile", "md_nccl"])
def test_sharded_masked_update_vs_fp64_learner(mgpu_runs, name, world):
    """A sharded masked update against the single-GPU fp64 learner on the global rollout (rank r holding global envs
    [r * n_envs, (r + 1) * n_envs)), two annealed updates with the Adam state carried: each rank's stored masks are the ones it fed
    at the right (env, t) rows and allow its actions; every rank's params and Adam state are bit-identical to rank 0's; params,
    Adam moments and all five losses match the learner, whose minibatches pair every sample with the mask of its own global row.
    World 1 runs the same cases on one GPU (no exchange)."""
    import mgpu_action_mask_worker as w
    assert (w.O, w.N_DISC, w.NVEC) == (O, N_DISC, NVEC)
    spec = w.CASES[name]
    if world == 1 and spec.get("p2p") is False:
        pytest.skip("the NCCL fallback exchanges between two or more ranks")
    out = mgpu_runs(world)
    ranks = [dict(np.load(os.path.join(out, f"{name}_r{r}.npz"))) for r in range(world)]
    r0 = ranks[0]
    what = f"{name} at world {world}"
    space = w.HEADS[spec["head"]]["action_space"]
    assert ("train_tile_kernel" if "PPO_DISABLE_FUSED" in spec.get("env", ()) else "train_fused_kernel") in str(r0["family_train"]), what
    Nl, T = spec["n_envs"], spec["n_steps"]
    for r, d in enumerate(ranks):
        assert not bool(d["comm_error"]), f"{what}: a peer-mailbox wait timed out on rank {r}"
        for t in ("params", "adam_m", "adam_v", "beta1_power", "beta2_power"):
            assert np.array_equal(d[t], r0[t]), f"{what}: rank {r} {t} differs from rank 0's"
        for u in range(spec["updates"]):
            fed = d[f"u{u}_fed_masks"].transpose(1, 0, 2).reshape(Nl * T, -1).astype(np.float32)  # flat row = env * n_steps + t
            assert np.array_equal(d[f"u{u}_action_masks"], fed), f"{what}: rank {r} update {u} stored other masks"
            assert allowed(d[f"u{u}_actions"], fed.astype(np.uint8), space), f"{what}: rank {r} took a forbidden action"
    ent, vf, clip, b1, b2, eps = r0["hparams"].astype(np.float64)
    h1, h2 = spec["hidden"]
    lay, P, _ = layout(space, h1, h2)
    loss = partial(learner_loss, activation=spec.get("activation", "tanh"), space=space, h1=h1, h2=h2, ent_coef=ent, vf_coef=vf)
    p0 = r0["p0"]
    p, state = p0, {}
    for u in range(spec["updates"]):
        bufs = {b: np.concatenate([d[f"u{u}_{b}"] for d in ranks], axis=0) for b in ("obs", "actions", "returns", "values", "neglogpacs")}
        bufs["actions"] = np.concatenate([bufs["actions"], np.concatenate([d[f"u{u}_action_masks"] for d in ranks], axis=0)], 1)
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
