"""Sharded multi-GPU updates against the fp64 learner, on the paths multi-GPU runs take.

One torch.distributed.run launch per world size W runs every case of mgpu_parity_worker.py (one process per GPU); the
worker writes what each rank holds, and this module computes the references and asserts.  The reference is learner_ref
and the loss_grad_ref functions of test_vf_clip_and_schedules and test_discrete, run on the global rollout (every rank's
rows, rank r holding global envs [r * n_envs, (r + 1) * n_envs)) with the permutations the cores report, the Adam state
carried from update to update.  Only the fixed rank-order sums differ from one GPU, so the single-GPU bars apply.

Per case: every rank's params, Adam moments and beta powers bit-identical to rank 0's; params, moments and losses against
the learner; the kernel families the case is meant to reach; no peer-mailbox timeout; graphs replayed, not rebuilt.  Per
epoch count: the permutations on every rank against glibc's random_shuffle, sharded and not.  The first rollout against a
single-GPU core of the global configuration (A, B, H) and the stepwise VecNormalize of the Discrete cases against the C
oracle.  W = 1 runs the same cases on one GPU (no exchange): it checks the harness and the references on any box."""
import os
import signal
import socket
import subprocess
import sys
from functools import partial

import numpy as np
import pytest

import oracle_lib as ol
import test_discrete as td
from conftest import ROOT, rel_err
from mgpu_parity_worker import CASES, PERM_CASES, SHUFFLE_SEED, SINGLE_GPU_ROLLOUT
from ppo_cpp_b200 import core
from ppo_cpp_b200 import meta_graph as mg
from ppo_cpp_b200.dist import shard_plan
from test_vf_clip_and_schedules import learner_ref, loss_grad_ref

WORLDS = (1, 2, 4, 8)
TRAIN_BUFS = ("obs", "actions", "returns", "values", "neglogpacs")
TIMEOUT = 1800
# the Adam moments against the learner's, tensor by tensor (max |got - want| / max |want|): at most 1.8e-5 measured over
# every case on one B200 (1000 W power limit), where the fp32 parameter trajectory drifting from the fp64 one dominates
ADAM_TOL = {"adam_m": 2e-4, "adam_v": 2e-4}


# ------------------------------------------------------------------ global rollout from the ranks' rows
def reassemble(per_rank):
    """Rank r's rollout_get rows are its envs in env-major order (row = env_local * n_steps + t) and it owns global envs
    [r * n_envs, (r + 1) * n_envs): the global env-major buffer is the ranks' rows one after the other."""
    return np.concatenate(per_rank, axis=0)


def rank_rows(global_rows, rank, world):
    """The rows of a global env-major buffer that rank `rank` of `world` produced."""
    n = global_rows.shape[0] // world
    return global_rows[rank * n:(rank + 1) * n]


def test_reassembly_matches_shard_plan():
    world, n_envs, n_steps, nmb, w = 4, 6, 5, 3, 3
    # rank r, local env e, step t, column j -> a value that names all four
    per_rank = [np.array([[1000 * r + 100 * e + t + 0.01 * j for j in range(w)] for e in range(n_envs) for t in range(n_steps)])
                for r in range(world)]
    g = reassemble(per_rank)
    plan = shard_plan(0, world, n_envs, n_steps, nmb)
    assert g.shape == (plan.n_batch_global, w)
    # the allgathered [rank][t][env_local] buffer the train kernels read, built from the ranks' own rows
    phys = np.concatenate([pr.reshape(n_envs, n_steps, w).transpose(1, 0, 2).reshape(-1, w) for pr in per_rank])
    for row in range(plan.n_batch_global):
        r = plan.owner_of_row(row, n_steps)
        env_local, t = divmod(row - r * n_envs * n_steps, n_steps)
        assert np.array_equal(g[row], per_rank[r][env_local * n_steps + t])
        assert np.array_equal(g[row], phys[plan.physical_row(row, n_steps)])
    for r in range(world):
        assert np.array_equal(rank_rows(g, r, world), per_rank[r])
        rows = [i for i in range(plan.n_batch_global) if plan.owner_of_row(i, n_steps) == r]
        assert np.array_equal(rank_rows(g, r, world), g[rows])


# ------------------------------------------------------------------ one launch per world size
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


_RUNS = {}


def _launch(world, out_dir):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "torch.distributed.run", "--nnodes", "1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
        "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "mgpu_parity_worker.py"), str(out_dir)]
    # its own session: on a timeout the whole process group goes, so no rank is left running
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, start_new_session=True)
    try:
        log, _ = p.communicate(timeout=TIMEOUT)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        log, _ = p.communicate()
        return False, f"timed out after {TIMEOUT} s\n{log[-6000:]}"
    return p.returncode == 0, log[-6000:]


@pytest.fixture(scope="module")
def mgpu(tmp_path_factory):
    """mgpu(W) -> the worker's output directory of world size W (launched on first use, once per module)."""
    import torch

    def get(world):
        if torch.cuda.device_count() < world:
            pytest.skip(f"needs {world} GPUs, the box has {torch.cuda.device_count()}")
        if world not in _RUNS:
            out = tmp_path_factory.mktemp(f"mgpu_w{world}")
            _RUNS[world] = (out,) + _launch(world, out)
        out, ok, log = _RUNS[world]
        assert ok, f"world {world}: the worker failed\n{log}"
        return out
    return get


def _load(out, name, world):
    return [dict(np.load(os.path.join(out, f"{name}_r{r}.npz"))) for r in range(world)]


# ------------------------------------------------------------------ expectations
def expected_families(name, world):
    """(substrings the train family must have, substrings it must not have, rollout family or None) of a case."""
    if name.startswith("G_"):
        base, p2p = name[2:], False
        base = "F_tanh" if base == "F" else base
    else:
        base, p2p = name, True
    persistent_rollout = "rollout_persistent_kernel (one cooperative launch per rollout)"
    per_step = "per-step kernels"
    if base in ("A", "B"):
        return (("train_umma_kernel", "persistent"), (), persistent_rollout) if p2p else (("train_umma_kernel",), ("persistent",), per_step)
    if base in ("C", "C_no_sq_ll"):
        return ("train_umma_kernel",), ("persistent",), persistent_rollout if p2p else per_step
    if base == "D":  # one GPU runs the single-CTA epoch kernel; a sharded run cannot
        return (("train_small_kernel", "persistent"), (), persistent_rollout) if world == 1 else (("train_small_kernel",), ("persistent",), persistent_rollout)
    if base == "E":
        return ("wgemm_kernel",), (), None if p2p else per_step
    if base in ("F_tanh", "F_relu"):
        return ("train_fused_kernel",), (), per_step
    if base == "F_tile":
        return ("train_tile_kernel",), (), per_step
    if base == "H":  # no tcgen05 family takes obs_dim 32: F or T, whichever the core selects
        return (), ("umma", "tcgen05", "wgemm"), persistent_rollout
    raise KeyError(name)


def _layout(spec):
    h1, h2 = spec["hidden"]
    space = spec.get("space", "box")
    lay = mg.param_layout(spec.get("obs_dim", 18), spec.get("act_dim", 18), h1, h2, action_space=space)
    names = [t for t in mg.TENSOR_ORDER[:mg.N_TRAINABLE_TENSORS] if t in lay]
    return [(t, slice(lay[t][0], lay[t][0] + int(np.prod(lay[t][1])))) for t in names], lay["model/q/w"][0]


def _loss_fn(spec, hp, cr_vf):
    h1, h2 = spec["hidden"]
    act = spec.get("activation", "tanh")
    if spec.get("space") == "discrete":
        return partial(td.loss_grad_ref, activation=act, h1=h1, h2=h2, ent_coef=hp[0], vf_coef=hp[1], o=spec.get("obs_dim", 18), n=spec.get("act_dim", 18))
    return partial(loss_grad_ref, mode=spec.get("vf", "shared"), cr_vf=cr_vf, h1=h1, h2=h2, ent_coef=hp[0], vf_coef=hp[1], activation=act)


def _check_replicas(ranks, what):
    for r, d in enumerate(ranks[1:], 1):
        for t in ("params", "adam_m", "adam_v", "beta1_power", "beta2_power"):
            assert np.array_equal(d[t], ranks[0][t]), f"{what}: rank {r} {t} differs from rank 0's"


# ------------------------------------------------------------------ the tests
@pytest.mark.gpu
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", sorted(CASES))
def test_sharded_update_vs_fp64_learner(mgpu, name, world):
    spec = CASES[name]
    if world == 1 and spec.get("p2p") is False:
        pytest.skip("the NCCL fallback exchanges between two or more ranks")
    ranks = _load(mgpu(world), name, world)
    r0 = ranks[0]
    what = f"{name} at world {world}"
    for r, d in enumerate(ranks):
        assert not bool(d["comm_error"]), f"{what}: a peer-mailbox wait timed out on rank {r}"
    fam_train, fam_rollout = str(r0["family_train"]), str(r0["family_rollout"])
    must, must_not, rollout = expected_families(name, world)
    assert all(s in fam_train for s in must) and not any(s in fam_train for s in must_not), (what, fam_train)
    assert rollout is None or fam_rollout == rollout, (what, fam_rollout)
    builds = r0["builds"].tolist()
    if spec.get("p2p") is False:
        assert builds == [0] * len(builds), (what, "NCCL inside a graph", builds)
    else:  # the schedule changes every update: the captured graphs are replayed, not rebuilt
        assert builds[0] > 0 and builds == [builds[0]] * len(builds), (what, builds)
    _check_replicas(ranks, what)

    hp = r0["hparams"].astype(np.float64)
    ent, vf, clip, b1, b2, eps = hp
    slices, P = _layout(spec)
    E, nmb = spec["epochs"], spec["nmb"]
    p0 = r0["p0"]
    p, state = p0, {}
    for u in range(spec["updates"]):
        bufs = {b: reassemble([d[f"u{u}_{b}"] for d in ranks]) for b in TRAIN_BUFS}
        perms = r0[f"u{u}_perms"]
        for r, d in enumerate(ranks):
            assert np.array_equal(d[f"u{u}_perms"], perms), f"{what}: rank {r} trained on other permutations"
        lr, cr, cr_vf = (float(x) for x in r0[f"u{u}_schedule"])
        loss = _loss_fn(spec, hp, cr_vf)
        learn = partial(learner_ref, nmb=nmb, lr=lr, cr=cr, loss_grad=loss, clip=clip, b1=b1, b2=b2, eps=eps, state=state)
        p, want = learn(p, bufs, perms)
        cols = slice(0, 5) if spec.get("space") == "discrete" else slice(0, 4)  # Box: clipfrac is a count of threshold tests
        got = r0[f"u{u}_losses"]
        assert np.allclose(got[cols], want[cols], rtol=2e-5, atol=1e-6), (what, f"update {u} losses", got, want)
        if f"u{u}_mb_ks" in r0:  # train_minibatch on the last epoch's permutation, the Adam state going on
            for k, got in zip(r0[f"u{u}_mb_ks"], r0[f"u{u}_mb_losses"]):
                p, want = learn(p, bufs, perms[-1:], ks=[int(k)])
                assert np.allclose(got[cols], want[cols], rtol=2e-5, atol=1e-6), (what, f"train_minibatch {k} losses", got, want)
    got = r0["params"]
    moved = np.abs(p[:P] - p0[:P]).max()
    diff = np.abs(got[:P] - p[:P]).max()
    adam = {key: max(rel_err(r0[key][sl], state[key[-1]][sl]) for _, sl in slices) for key in ADAM_TOL}
    print(f"{what}: train {fam_train.split(' ')[0]}{' (persistent)' if 'persistent' in fam_train else ''}, "
          f"rollout {fam_rollout.split(' ')[0]}, param diff / moved = {diff / moved:.3e}, "
          f"adam_m {adam['adam_m']:.2e}, adam_v {adam['adam_v']:.2e}")
    assert diff < max(5e-4, 4e-5 * E * nmb) * moved, (what, "params", diff / moved)
    assert np.array_equal(got[P:], p0[P:])
    for key in ADAM_TOL:
        for t, sl in slices:
            err = rel_err(r0[key][sl], state[key[-1]][sl])
            assert err < ADAM_TOL[key], (what, key, t, err)
    assert float(r0["beta1_power"][0]) == pytest.approx(state["b1p"], rel=1e-5)
    assert float(r0["beta2_power"][0]) == pytest.approx(state["b2p"], rel=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", sorted(PERM_CASES))
def test_sharded_permutations_equal_glibc_shuffle(mgpu, name, world):
    """Every rank's permutations are std::srand(seed) + std::random_shuffle compounded over the epochs of an update, with
    the epochs built on different ranks and exchanged (also when there are fewer epochs than ranks) and without; the
    second update restarts from the identity and goes on with the rand() stream."""
    spec = PERM_CASES[name]
    ranks = _load(mgpu(world), name, world)
    E = spec["epochs"]
    n = spec["n_envs"] * spec["n_steps"] * world
    want0 = core.host_random_shuffle(SHUFFLE_SEED, n, E)
    stream = core.host_rand(SHUFFLE_SEED, 2 * E * (n - 1))[E * (n - 1):]
    a = np.arange(n, dtype=np.int32)
    want1 = []
    k = 0
    for e in range(E):
        for i in range(1, n):
            j = int(stream[k]) % (i + 1)
            k += 1
            a[i], a[j] = a[j], a[i]
        want1.append(a.copy())
    for r, d in enumerate(ranks):
        assert not bool(d["comm_error"]), (name, world, r)
        assert np.array_equal(d["u0_perms"], want0), f"{name} at world {world}: rank {r}, update 0"
        assert np.array_equal(d["u1_perms"], np.stack(want1)), f"{name} at world {world}: rank {r}, update 1"


@pytest.mark.gpu
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", SINGLE_GPU_ROLLOUT)
def test_sharded_rollout_equals_single_gpu(mgpu, name, world):
    """The first rollout: each rank's rows are those of one GPU running every global env (same Philox stream per global env,
    VecNormalize moments summed over the ranks), and the normalisation counts are equal."""
    ranks = _load(mgpu(world), name, world)
    r0 = ranks[0]
    for b in ("obs", "actions", "values", "neglogpacs", "returns", "dones"):
        single = r0[f"single_{b}"]
        for r, d in enumerate(ranks):
            mine = rank_rows(single, r, world)
            if b == "dones":
                assert np.array_equal(d[f"u0_{b}"], mine), (name, world, r, b)
            else:
                assert rel_err(d[f"u0_{b}"], mine) < 2e-5, (name, world, r, b, rel_err(d[f"u0_{b}"], mine))
    for r, d in enumerate(ranks):
        assert d["stats0_obs_count"] == r0["single_stats_obs_count"] and d["stats0_ret_count"] == r0["single_stats_ret_count"], (name, world, r)
        for k in ("obs_mean", "obs_var", "ret_var"):
            assert rel_err(d[f"stats0_{k}"], r0[f"single_stats_{k}"]) < 1e-5, (name, world, r, k)


@pytest.mark.gpu
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", ["F_tanh", "G_F"])
def test_sharded_vecnorm_equals_oracle(mgpu, name, world):
    """The stepwise VecNormalize of a host-env rollout on every rank (moments summed over the ranks: over the mailbox with
    peer access, by ncclAllReduce without) against the C oracle's VecNormalize over all global envs."""
    if world == 1 and name == "G_F":
        pytest.skip("the NCCL fallback exchanges between two or more ranks")
    ranks = _load(mgpu(world), name, world)
    r0 = ranks[0]
    raw, rew, done, obs0 = r0["traj_raw"], r0["traj_rew"], r0["traj_done"], r0["traj_obs0"]
    N, O = obs0.shape
    lib = ol.load()
    vn = lib.oracle_vecnorm_create(N, O, 1)
    try:
        lib.oracle_vecnorm_reset_f32(vn, obs0, np.zeros((N, O), np.float32))
        out_obs, out_rew = np.zeros((N, O), np.float32), np.zeros(N, np.float32)
        for u in range(raw.shape[0]):
            for t in range(raw.shape[1]):
                lib.oracle_vecnorm_step_f32(vn, np.ascontiguousarray(raw[u, t]), np.ascontiguousarray(rew[u, t]),
                                            np.ascontiguousarray(done[u, t]), out_obs, out_rew)
        v = vn.contents
        want = dict(obs_count=v.obs_rms.count, ret_count=v.ret_rms.count, obs_mean=np.ctypeslib.as_array(v.obs_rms.mean, (O,)).copy(),
                    obs_var=np.ctypeslib.as_array(v.obs_rms.var, (O,)).copy(), ret_var=np.ctypeslib.as_array(v.ret_rms.var, (1,)).copy())
    finally:
        lib.oracle_vecnorm_destroy(vn)
    for r, d in enumerate(ranks):
        assert d["stats_obs_count"] == want["obs_count"] and d["stats_ret_count"] == want["ret_count"], (name, world, r)
        for k in ("obs_mean", "obs_var", "ret_var"):
            assert rel_err(d[f"stats_{k}"], want[k]) < 1e-5, (name, world, r, k, rel_err(d[f"stats_{k}"], want[k]))
