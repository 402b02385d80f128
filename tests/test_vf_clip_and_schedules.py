"""Stable-Baselines' three value losses (cliprange_vf None / < 0 / >= 0, ppo_vf_clip) and per-update schedules of lr,
cliprange and cliprange_vf on device-resident scalars.

The reference for the losses is an independent fp64 PyTorch autograd restatement of Stable-Baselines' PPO2 loss, with
TensorFlow's tie rules written out (Maximum's gradient goes to its first operand on >=, clip_by_value passes it on
-b <= x <= b; torch.maximum would split a tie 0.5 / 0.5).  CPU tests: the reference and its tie fixture, and the two graph
readers.  GPU tests: every kernel family, whole updates, schedules replaying the captured graphs, the host C++ PPO2.
test_multi_gpu_parity.py runs the same learner on sharded multi-GPU updates."""
import os
import subprocess
from functools import partial

import numpy as np
import pytest
import torch

from conftest import ROOT, load_weights, rel_err
from ppo_cpp_b200 import meta_graph as mg

HALF_LOG_2PI = 0.9189385175704956
HALF_LOG_2PIE = 1.4189385175704956
TOL = 1e-5


# ------------------------------------------------------------------ fp64 reference (PyTorch autograd)
def _layout(h1, h2, O=18, A=18):
    lay = mg.param_layout(O, A, h1, h2)
    return [lay[n] for n in mg.TENSOR_ORDER[:13]], lay["model/q/w"][0]


def _tf_max(x, y):
    """max(x, y) with TensorFlow's gradient: all of it to x where x >= y."""
    return torch.where(x >= y, x, y)


def _tf_clip(x, lo, hi):
    """clip_by_value = maximum(minimum(x, hi), lo): Minimum passes to x on x <= hi, Maximum on min(x, hi) >= lo."""
    t = torch.where(x <= hi, x, hi)
    return torch.where(t >= lo, t, lo)


def _act(name, mask="gt"):
    """The hidden-layer activation; ReLU's gradient masks on output > 0 (TensorFlow's ReluGrad, mask="gt") or, to show that a
    fixture tells the two apart, on input >= 0 (mask="ge": a unit at exactly 0 passes it)."""
    if name == "tanh":
        return torch.tanh
    if mask == "gt":
        return torch.relu
    return lambda z: torch.where(z >= 0, z, torch.zeros_like(z))


def value_loss(v, old_v, R, mode, cr, cr_vf, tie="tf"):
    """Per-sample max(l1, l2) of Stable-Baselines' ppo2.py for ppo_vf_clip `mode`; tie="split" gives torch's own
    0.5 / 0.5 rule (used only to show that a fixture tells the two apart)."""
    if mode == "none":
        vc = v
    else:
        b = torch.tensor(cr if mode == "shared" else cr_vf, dtype=torch.float64)
        dvo = v - old_v
        vc = old_v + (_tf_clip(dvo, -b, b) if tie == "tf" else torch.clamp(dvo, -b, b))
    l1, l2 = (v - R) ** 2, (vc - R) ** 2
    return _tf_max(l1, l2) if tie == "tf" else torch.maximum(l1, l2)


def loss_grad_ref(params, obs, act, adv, ret, old_nlp, old_v, cr, mode="shared", cr_vf=0.0, h1=4, h2=5,
                  ent_coef=0.0007160293171182275, vf_coef=0.5, tie="tf", activation="tanh", mask="gt"):
    """fp64 loss + gradient of the 13 trainable tensors (graph gradient order) and the five reported losses of a Gaussian
    policy; the observation and action widths are those of obs and act."""
    lay, P = _layout(h1, h2, np.shape(obs)[1], np.shape(act)[1])
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
    vf = 0.5 * value_loss(v, ov, R, mode, cr, cr_vf, tie).mean()
    ent = (ls + HALF_LOG_2PIE).sum()
    loss = pg - ent * ent_coef + vf * vf_coef
    loss.backward()
    with torch.no_grad():
        kl = 0.5 * ((nlp - onl) ** 2).mean()
        cf = ((ratio - 1.0).abs() > cr).double().mean()
    losses = np.array([pg.item(), vf.item(), ent.item(), kl.item(), cf.item()])
    return p.grad.numpy().copy(), losses


def tie_fixture(rng, B, cr_vf, v0=0.25):
    """Value targets around a value head that outputs exactly v0 (zero value weights): v - old_v = +-cr_vf exactly, and
    (v - R)^2 == (vc - R)^2 with v - old_v outside the range, mixed with plain samples.  All dyadic, exact in fp32 and fp64."""
    assert cr_vf == 0.125 and v0 == 0.25
    old_v = rng.standard_normal(B) * 0.3
    R = rng.standard_normal(B) * 0.3
    kinds = rng.integers(0, 5, B)
    for i, k in enumerate(kinds):
        if k == 0:  # upper clip bound hit exactly
            old_v[i] = v0 - cr_vf
        elif k == 1:  # lower bound
            old_v[i] = v0 + cr_vf
        elif k == 2:  # l1 == l2, clipped from above: vc = 0.125, R midway
            old_v[i], R[i] = 0.0, 0.1875
        elif k == 3:  # l1 == l2, clipped from below: vc = 0.375
            old_v[i], R[i] = 0.5, 0.3125
    return old_v.astype(np.float32), R.astype(np.float32)


def synth_batch(rng, params, h1, h2, B, O=18, A=18):
    lay, P = _layout(h1, h2)
    p = params.astype(np.float64)
    t = [p[o:o + int(np.prod(s))].reshape(s) for o, s in lay]
    obs = rng.standard_normal((B, O)).astype(np.float32)
    x = obs.astype(np.float64)
    mu = np.tanh(np.tanh(x @ t[0] + t[1]) @ t[4] + t[5]) @ t[10] + t[11]
    v = (np.tanh(np.tanh(x @ t[2] + t[3]) @ t[6] + t[7]) @ t[8] + t[9])[:, 0]
    std = np.exp(t[12].ravel())
    act = (mu + std * rng.standard_normal((B, A))).astype(np.float32)
    z = (act - mu) / std
    old_nlp = (0.5 * (z * z).sum(1) + A * HALF_LOG_2PI + np.log(std).sum() + 0.1 * rng.standard_normal(B)).astype(np.float32)
    old_v = (v + 0.3 * rng.standard_normal(B)).astype(np.float32)
    # returns off the value by a common bias: the value-bias gradient sum(dL/dv) is then not a near-cancelling sum
    ret = (v + 0.3 + 0.5 * rng.standard_normal(B)).astype(np.float32)
    adv = rng.standard_normal(B).astype(np.float32)
    return obs, act, adv, ret, old_nlp, old_v


def rand_params(rng, h1, h2, A=18):
    _, P = _layout(h1, h2)
    Pq = mg.param_layout(18, A, h1, h2)["__total__"][0]
    p = (rng.standard_normal(Pq) * min(0.3, 1.5 / np.sqrt(max(h1, h2)))).astype(np.float32)
    lay = mg.param_layout(18, A, h1, h2)
    o = lay["model/pi/logstd"][0]
    p[o:o + A] = (-0.5 + 0.2 * rng.standard_normal(A)).astype(np.float32)
    return p


def tie_params(rng, h1, h2, v0=0.25):
    """Random policy, value head of zero weights and bias v0: every family computes v = v0 exactly."""
    p = rand_params(rng, h1, h2)
    lay = mg.param_layout(18, 18, h1, h2)
    o = lay["model/vf/w"][0]
    p[o:o + h2] = 0.0
    p[lay["model/vf/b"][0]] = v0
    return p


def tensor_slices(h1, h2):
    lay, _ = _layout(h1, h2)
    return [slice(o, o + int(np.prod(s))) for o, s in lay]


# ------------------------------------------------------------------ CPU: the reference
def test_reference_value_loss_matches_closed_form():
    """The autograd value loss against the per-sample closed form the kernels evaluate (value_loss_term in
    device_common.cuh), in fp64, for all three modes."""
    rng = np.random.default_rng(1)
    n = 4000
    v, ov, R = (rng.standard_normal(n) for _ in range(3))
    cr, cr_vf = 0.2, 0.35
    for mode in ("shared", "none", "separate"):
        vt = torch.tensor(v, requires_grad=True)
        l = value_loss(vt, torch.tensor(ov), torch.tensor(R), mode, cr, cr_vf)
        l.sum().backward()
        r = cr_vf if mode == "separate" else cr
        dvo = v - ov
        vc = v if mode == "none" else ov + np.maximum(np.minimum(dvo, r), -r)
        l1, l2 = (v - R) ** 2, (vc - R) ** 2
        tk = l1 >= l2
        inr = np.ones(n, bool) if mode == "none" else (dvo <= r) & (dvo >= -r)
        assert np.array_equal(l.detach().numpy(), np.where(tk, l1, l2))
        assert np.allclose(vt.grad.numpy(), np.where(tk, 2 * (v - R), np.where(inr, 2 * (vc - R), 0.0)), rtol=1e-14, atol=1e-14)


def test_tie_fixture_is_discriminating():
    """On the tie fixture TensorFlow's rule and a 0.5 / 0.5 split give different value-head gradients in SEPARATE mode, so
    a kernel that passes the GPU comparison below implements TF's rule; the random batch alone would not tell them apart."""
    rng = np.random.default_rng(7)
    B = 512
    p = tie_params(rng, 4, 5)
    obs, act, adv, ret, old_nlp, _ = synth_batch(rng, p, 4, 5, B)
    old_v, R = tie_fixture(rng, B, 0.125)
    sl = tensor_slices(4, 5)
    g_tf, _ = loss_grad_ref(p, obs, act, adv, R, old_nlp, old_v, 0.2, "separate", 0.125)
    g_split, _ = loss_grad_ref(p, obs, act, adv, R, old_nlp, old_v, 0.2, "separate", 0.125, tie="split")
    for t in (8, 9):  # vf/w, vf/b: apart by far more than the 1e-5 bar of the GPU comparison
        assert rel_err(g_split[sl[t]], g_tf[sl[t]]) > 100 * TOL, t
    # and the modes differ from each other on it (the range matters, and NONE is not SEPARATE)
    g_sh, _ = loss_grad_ref(p, obs, act, adv, R, old_nlp, old_v, 0.2, "shared", 0.125)
    g_no, _ = loss_grad_ref(p, obs, act, adv, R, old_nlp, old_v, 0.2, "none", 0.125)
    assert rel_err(g_sh[sl[9]], g_tf[sl[9]]) > 100 * TOL and rel_err(g_no[sl[9]], g_tf[sl[9]]) > 100 * TOL


# ------------------------------------------------------------------ CPU: the graph readers
def _graph(tmp_path, vf_clip, name=None):
    tensors, _ = load_weights("graph_4_5_init.npz")
    path = str(tmp_path / (name or f"g_{vf_clip}.meta.txt"))
    mg.write_meta_txt(path, tensors, ent_coef=0.0007160293171182275, vf_clip=vf_clip)
    return path


@pytest.mark.parametrize("vf_clip", [None, "shared", "none", "separate"])
def test_readers_classify_the_value_loss(tmp_path, vf_clip):
    from ppo_cpp_b200 import core
    path = _graph(tmp_path, vf_clip)
    want = vf_clip or "shared"  # no loss sub-graph: the shipped graph's form
    assert mg.parse_meta_txt(path).vf_clip == want
    assert core.meta_vf_clip(path) == want
    info, params = core.meta_parse(path)
    assert (info.hidden1, info.hidden2) == (4, 5)


@pytest.mark.parametrize("edit", ["bound", "operand", "square"])
def test_readers_reject_an_unknown_value_loss(tmp_path, edit):
    from ppo_cpp_b200 import core
    path = _graph(tmp_path, "separate")
    text = open(path, encoding="latin-1").read()
    if edit == "bound":  # clip_by_value(x, -vf_range, policy range): neither form
        old = '    name: "loss/clip_by_value/Minimum"\n    op: "Minimum"\n    input: "loss/sub"\n    input: "loss/clip_range_vf_ph"\n'
        new = old.replace('input: "loss/clip_range_vf_ph"', 'input: "loss/clip_range_ph"')
    elif edit == "operand":  # vpred_clipped = vpred + clip(...)
        old = '    op: "Add"\n    input: "loss/old_vpred_ph"\n'
        new = '    op: "Add"\n    input: "train_model/strided_slice"\n'
    else:  # max(square(...), abs(...))
        old = '    name: "loss/Square_2"\n    op: "Square"\n'
        new = '    name: "loss/Square_2"\n    op: "Abs"\n'
    assert text.count(old) == 1
    with open(path, "w", encoding="latin-1") as f:
        f.write(text.replace(old, new))
    with pytest.raises(ValueError):
        mg.parse_meta_txt(path)
    with pytest.raises(core.PPOError, match=r"\[-4\]"):
        core.meta_vf_clip(path)
    with pytest.raises(core.PPOError, match=r"\[-4\]"):
        core.meta_parse(path)


# ------------------------------------------------------------------ GPU: loss + gradient of every family
FAMILIES = [  # (h, B, env switch, family marker)
    (4, 2048, None, "small"), (4, 77, None, "small"),
    (64, 1000, None, "tcgen05"), (64, 20000, None, "tcgen05"),
    (64, 1000, "PPO_DISABLE_UMMA", "fused"), (64, 1000, "PPO_DISABLE_FUSED", "tile"),
    (128, 300, None, "tcgen05"), (256, 1000, None, "tcgen05"), (256, 77, None, "tcgen05"),
]


def _family_core(core_mod, monkeypatch, h, env, p):
    if env:
        monkeypatch.setenv(env, "1")
    c = core_mod.PPOCore(hidden1=h, hidden2=5 if h == 4 else h, n_envs=4, n_steps=8, nminibatches=4)
    if env:
        monkeypatch.delenv(env)
    c.set_tensor("params", p)
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("h,B,env,fam", FAMILIES)
def test_loss_grad_vf_every_family_vs_fp64(monkeypatch, h, B, env, fam):
    from ppo_cpp_b200 import core as core_mod
    h2 = 5 if h == 4 else h
    rng = np.random.default_rng(100 + h + B)
    sl = tensor_slices(h, h2)
    c = _family_core(core_mod, monkeypatch, h, env, rand_params(rng, h, h2))
    assert fam in c.kernel_family("train"), c.kernel_family("train")
    for fixture in ("random", "ties"):
        p = rand_params(rng, h, h2) if fixture == "random" else tie_params(rng, h, h2)
        c.set_tensor("params", p)
        obs, act, adv, ret, old_nlp, old_v = synth_batch(rng, p, h, h2, B)
        if fixture == "ties":
            old_v, ret = tie_fixture(rng, B, 0.125)
        # SHARED through the new entry is the old entry, bit for bit
        c.vf_clip = "shared"
        g_old, l_old = c.loss_grad(obs, act, adv, ret, old_nlp, old_v, 0.2)
        g_new, l_new = c.loss_grad(obs, act, adv, ret, old_nlp, old_v, 0.2, cliprange_vf=0.125)
        assert np.array_equal(g_old, g_new) and np.array_equal(l_old, l_new)
        for mode in ("none", "separate"):
            c.vf_clip = mode
            g, l = c.loss_grad(obs, act, adv, ret, old_nlp, old_v, 0.2, cliprange_vf=0.125)
            g64, l64 = loss_grad_ref(p, obs, act, adv, ret, old_nlp, old_v, 0.2, mode, 0.125, h1=h, h2=h2)
            for t in range(13):
                assert rel_err(g[sl[t]], g64[sl[t]]) < TOL, (fixture, mode, t, rel_err(g[sl[t]], g64[sl[t]]))
            assert np.allclose(l[:4], l64[:4], rtol=TOL, atol=1e-7), (fixture, mode, l, l64)
            assert l[4] == pytest.approx(l64[4], abs=1.5 / B)
    c.close()


@pytest.mark.gpu
def test_separate_mode_needs_cliprange_vf():
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(5)
    c = core_mod.PPOCore(n_envs=4, n_steps=8, nminibatches=4)
    p = rand_params(rng, 4, 5)
    c.set_tensor("params", p)
    obs, act, adv, ret, old_nlp, old_v = synth_batch(rng, p, 4, 5, 32)
    c.vf_clip = "separate"
    assert c.vf_clip == "separate"
    with pytest.raises(core_mod.PPOError, match="needs cliprange_vf"):
        c.loss_grad(obs, act, adv, ret, old_nlp, old_v, 0.2)
    with pytest.raises(core_mod.PPOError, match=r"\[-1\]"):
        c.loss_grad(obs, act, adv, ret, old_nlp, old_v, 0.2, cliprange_vf=-1.0)
    c.synth_env_reset()
    c.rollout_synthetic()
    with pytest.raises(core_mod.PPOError, match="needs cliprange_vf"):
        c.train_update(3e-4, 0.2)
    with pytest.raises(ValueError):
        c.vf_clip = "clipped"
    c.close()


# ------------------------------------------------------------------ GPU: whole updates against an fp64 learner
def learner_ref(flat, bufs, perms, nmb, lr, cr, loss_grad, clip=0.5, b1=0.9, b2=0.999, eps=1e-5, state=None, ks=None):
    """PPO2::learn's epoch / minibatch loop (ppo2.hpp:264-335) on one rollout in fp64: per-minibatch advantage
    normalisation, loss gradient, clip_by_global_norm and TF's ApplyAdam, on the core's own permutations.

    loss_grad(params, obs, actions, advs, returns, old_neglogp, old_values, cliprange) -> (gradient of the trainable
    parameters, five losses) is loss_grad_ref, or test_discrete's for a categorical head, bound to the net with
    functools.partial.  state: the Adam moments and beta powers {"m", "v", "b1p", "b2p"} to start from (absent: zero
    moments and powers b1, b2, a fresh core), updated in place, so that a chain of calls is a chain of updates.  ks: the
    minibatches of each epoch to run (all of them by default; a train_minibatch call is one)."""
    st = {} if state is None else state
    p = flat.astype(np.float64).copy()
    m, v = st.get("m"), st.get("v")
    b1p, b2p = st.get("b1p", b1), st.get("b2p", b2)
    nb = bufs["obs"].shape[0]
    Bm = nb // nmb
    rows = []
    for perm in perms:
        src = np.empty_like(perm)
        src[perm] = np.arange(nb)  # Eigen's perm * buf writes row i to slot perm[i] (ppo2.hpp:291-296)
        for k in (range(nmb) if ks is None else ks):
            idx = src[k * Bm:(k + 1) * Bm]
            ret, val = bufs["returns"][idx, 0], bufs["values"][idx, 0]
            a = ret.astype(np.float64) - val
            adv = (a - a.mean()) / (np.sqrt(((a - a.mean()) ** 2).mean()) + 1e-8)
            g, l = loss_grad(p, bufs["obs"][idx], bufs["actions"][idx], adv, ret, bufs["neglogpacs"][idx, 0], val, cr)
            rows.append(l)
            if m is None:
                m, v = np.zeros_like(g), np.zeros_like(g)
            gn = np.sqrt((g * g).sum())
            g = g * clip * min(1.0 / gn, 1.0 / clip)
            m += (g - m) * (1 - b1)
            v += (g * g - v) * (1 - b2)
            p[:g.size] -= lr * np.sqrt(1 - b2p) / (1 - b1p) * m / (np.sqrt(v) + eps)
            b1p *= b1
            b2p *= b2
    st.update(m=m, v=v, b1p=b1p, b2p=b2p)
    return p, np.mean(rows, axis=0)


UPDATE_CASES = [  # (h1, h2, n_envs, n_steps, nmb, epochs, family marker)
    (4, 5, 1, 2048, 32, 2, "small"),           # C1's shape: the single-CTA S epoch kernel
    (64, 64, 1024, 16, 2, 2, "persistent"),    # C3's minibatch (8192 samples) on the persistent U epoch kernel
    (256, 256, 128, 32, 1, 1, "tcgen05"),      # a [256,256] update on W
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["none", "separate"])
@pytest.mark.parametrize("h1,h2,n_envs,n_steps,nmb,epochs,fam", UPDATE_CASES)
def test_train_update_vf_vs_fp64_learner(mode, h1, h2, n_envs, n_steps, nmb, epochs, fam):
    from ppo_cpp_b200 import core as core_mod
    rng = np.random.default_rng(21)
    ent = 0.0007160293171182275
    flat = load_weights("graph_4_5_init.npz")[1] if h1 == 4 else rand_params(rng, h1, h2)
    c = core_mod.PPOCore(hidden1=h1, hidden2=h2, n_envs=n_envs, n_steps=n_steps, nminibatches=nmb, noptepochs=epochs, ent_coef=ent, seed=9)
    c.set_tensor("params", flat)
    fam_name = c.kernel_family("train")
    assert fam in fam_name, fam_name
    c.vf_clip = mode
    c.synth_env_reset()
    c.rollout_synthetic()
    bufs = {n: c.rollout_get(n) for n in ("obs", "actions", "returns", "values", "neglogpacs")}
    c.shuffle_seed(42)
    losses = c.train_update(3.9e-4, 0.2, cliprange_vf=0.1)
    perms = [c.train_get_permutation(e) for e in range(epochs)]
    got = c.get_tensor("params")
    c.close()
    p64, want = learner_ref(flat, bufs, perms, nmb, 3.9e-4, 0.2, partial(loss_grad_ref, mode=mode, cr_vf=0.1, h1=h1, h2=h2, ent_coef=ent))
    _, P = _layout(h1, h2)
    moved = np.abs(p64[:P] - flat[:P]).max()
    print(f"{mode} [{h1},{h2}] on {fam_name}: param diff / moved = {np.abs(got[:P] - p64[:P]).max() / moved:.3e}")
    # the bar of test_train_update_vs_oracle_learner (fp32 oracle), here against fp64
    assert np.abs(got[:P] - p64[:P]).max() < max(5e-4, 4e-5 * epochs * nmb) * moved
    assert np.allclose(losses[:4], want[:4], rtol=2e-5, atol=1e-6), (losses, want)
    assert np.array_equal(got[P:], flat[P:])


# ------------------------------------------------------------------ GPU: schedules replay the captured graphs
def _schedule_run(core_mod, monkeypatch, env, h, n_envs, n_steps, nmb, epochs, mode):
    for e in env:
        monkeypatch.setenv(e, "1")
    c = core_mod.PPOCore(hidden1=h, hidden2=5 if h == 4 else h, n_envs=n_envs, n_steps=n_steps, nminibatches=nmb, noptepochs=epochs, seed=4)
    for e in env:
        monkeypatch.delenv(e)
    c.init_orthogonal(3)
    c.vf_clip = mode
    c.shuffle_seed(17)
    c.synth_env_reset()
    losses, builds = [], []
    n_updates = 4
    for update in range(1, n_updates + 1):
        frac = 1.0 - (update - 1) / n_updates  # Stable-Baselines' schedule argument
        c.rollout_synthetic()
        losses.append(c.train_update(3e-4 * frac, 0.2 * frac + 0.05, cliprange_vf=0.3 * frac))
        builds.append(c.graph_builds())
    params = c.get_tensor("params")
    ctr, rollout = c.counters(), c.kernel_family("rollout")
    c.close()
    return np.array(losses), params, builds, ctr, rollout


@pytest.mark.gpu
@pytest.mark.parametrize("shuffle", ["gpu", "host"])
@pytest.mark.parametrize("h,n_envs,n_steps,nmb,epochs,mode,env", [
    pytest.param(64, 256, 32, 4, 2, "separate", [], id="64-256-32-4-2-separate"),
    pytest.param(4, 8, 64, 4, 2, "none", [], id="4-8-64-4-2-none"),
    pytest.param(256, 64, 32, 2, 2, "separate", [], id="256-64-32-2-2-separate"),
    # U per minibatch (train_step_device) and the per-step rollout, captured as one graph
    pytest.param(64, 256, 32, 4, 2, "separate", ["PPO_DISABLE_PERSISTENT"], id="64-256-32-4-2-separate-PPO_DISABLE_PERSISTENT")])
def test_annealed_updates_replay_graphs_and_equal_eager(monkeypatch, shuffle, h, n_envs, n_steps, nmb, epochs, mode, env):
    """lr, cliprange and cliprange_vf change every update: the captured graphs are replayed, not rebuilt (the graph count
    stays at its value after the first update), and the run equals the same launches made without graphs bit for bit.
    A replayed graph counts the kernels and copies it holds, so both runs report the same work."""
    from ppo_cpp_b200 import core as core_mod
    base = env + (["PPO_DISABLE_GPU_SHUFFLE"] if shuffle == "host" else [])
    l_g, p_g, builds, ctr_g, rollout = _schedule_run(core_mod, monkeypatch, base, h, n_envs, n_steps, nmb, epochs, mode)
    l_e, p_e, builds_e, ctr_e, _ = _schedule_run(core_mod, monkeypatch, base + ["PPO_DISABLE_GRAPH"], h, n_envs, n_steps, nmb, epochs, mode)
    assert builds[0] > 0 and builds == [builds[0]] * len(builds), builds
    assert builds_e == [0] * len(builds_e)
    assert np.all(np.isfinite(l_g))
    assert np.array_equal(l_g, l_e) and np.array_equal(p_g, p_e)
    assert ctr_g["graph_launches"] > 0 and ctr_e["graph_launches"] == 0
    for k in ("kernel_launches", "h2d_bytes", "d2h_bytes"):
        assert ctr_g[k] == ctr_e[k], (k, ctr_g, ctr_e)
    # the synthetic rollout is captured as a graph only where it runs as per-step kernels
    assert (rollout == "per-step kernels") == (h == 256 or "PPO_DISABLE_PERSISTENT" in env), rollout


# ------------------------------------------------------------------ GPU: the host C++ PPO2 and its CLI
@pytest.mark.gpu
def test_host_ppo2_cliprange_vf(tmp_path):
    host = os.path.join(ROOT, "ppo_cpp_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    exe = os.path.join(host, "bin", "ppo_cpp")

    def run(graph, *extra):
        cmd = [exe, "-d", str(tmp_path / "exp"), "--graph_path", graph, "--steps", "4096", "--lr", "0.00039", "--cr", "0.161",
               "--num_epochs", "2", "--batch_steps", "1024", "--threads", "2", "--seed", "5", "--saves", "1", *extra]
        return subprocess.run(cmd, capture_output=True, text=True, timeout=300)

    sep = _graph(tmp_path, "separate")
    r = run(sep, "--cliprange_vf", "0.3")
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    rows = [l for l in r.stdout.splitlines() if l.count(",") == 6 and l.endswith(",")]
    assert len(rows) == 2 and "cliprange_vf is ignored" not in r.stdout
    r = run(sep)  # the default -1
    assert r.returncode != 0 and "cliprange_vf must be >= 0" in r.stderr, r.stdout[-2000:] + r.stderr[-2000:]
    r = run(_graph(tmp_path, "none"), "--cliprange_vf", "0.3")
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "cliprange_vf is ignored: the graph does not clip the value" in r.stdout
