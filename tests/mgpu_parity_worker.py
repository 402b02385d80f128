"""Worker of test_multi_gpu_parity.py: one process per GPU under torch.distributed.run,
    python -m torch.distributed.run --nnodes 1 --nproc-per-node W --master-addr 127.0.0.1 --master-port P \\
        tests/mgpu_parity_worker.py OUT_DIR
Runs every case of CASES and PERM_CASES on sharded cores and writes what each rank holds to OUT_DIR/<case>_r<rank>.npz: its
own rollout rows of every update, the permutations, params, Adam state, losses, kernel families and graph build counts.
It computes no reference and asserts nothing; the test does both, so that a failure names the case and the quantity."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppo_cpp_b200 import core  # noqa: E402
from ppo_cpp_b200.dist import env_world, setup_comm  # noqa: E402

ENT = 0.01  # large enough that the entropy term moves logstd (Box) and the logits (Discrete) next to the surrogate
BUFS = ("obs", "actions", "returns", "values", "neglogpacs", "dones")
# Per-rank sizes; the global run is W times as many envs.  updates: rollout + train_update pairs with an annealed schedule.
_A = dict(hidden=(64, 64), n_envs=1024, n_steps=16, nmb=4, epochs=2, updates=3)
_C = dict(hidden=(64, 64), n_envs=48, n_steps=32, nmb=4, epochs=2, updates=2)
_E = dict(hidden=(256, 256), n_envs=64, n_steps=16, nmb=2, epochs=2, updates=2)
_F = dict(hidden=(64, 64), space="discrete", n_envs=128, n_steps=16, nmb=4, epochs=2, updates=2)
CASES = {
    # C3's path: persistent U epoch kernel, gradients summed over the peer mailbox; two train_minibatch calls (the
    # cooperative per-minibatch kernel) after the second update continue the same mailbox sequence numbers
    "A": dict(_A, minibatches_after=(1, (1, 3))),
    # 3 100 samples per rank-minibatch: 24 full tiles and a ragged one, ReLU template, cliprange_vf
    "B": dict(_A, n_envs=775, activation="relu", vf="separate"),
    "C": _C,                                          # U per minibatch + grad_reduce_adam_coop_kernel
    "C_no_sq_ll": dict(_C, env=("PPO_DISABLE_SQ_LL",)),  # ... with the grid barrier instead of the LL sum-of-squares words
    "D": dict(_C, hidden=(4, 5)),                     # S per minibatch + coop kernel
    "E": _E,                                          # W + grad_reduce_adam_big_kernel
    "F_tanh": _F,                                     # categorical head on F, stepwise VecNormalize
    "F_relu": dict(_F, activation="relu"),
    "F_tile": dict(_F, env=("PPO_DISABLE_FUSED",)),   # ... on T
    # the NCCL fallback: ncclAllReduce of gradients and moments, sqnorm_kernel + adam_kernel, no graphs
    "G_A": dict(_A, updates=2, p2p=False),
    "G_C": dict(_C, p2p=False),
    "G_E": dict(_E, p2p=False),
    "G_F": dict(_F, p2p=False),
    # the largest VecNormalize moment payload of the mailbox (obs_dim = act_dim = 32) in the persistent rollout
    "H": dict(_C, obs_dim=32, act_dim=32),
}
# global single-GPU rollouts to compare the sharded first rollout with
SINGLE_GPU_ROLLOUT = ("A", "B", "H")
PERM_CASES = {f"perm_e{e}{'_unsharded' if u else ''}": dict(hidden=(4, 5), n_envs=48, n_steps=32, nmb=4, epochs=e, updates=2,
                                                             env=("PPO_DISABLE_SHUFFLE_SHARDING",) if u else ())
              for e in (1, 3, 10) for u in (False, True)}
SHUFFLE_SEED = 42


def schedule(spec, u):
    """lr, cliprange and cliprange_vf of update u, annealed as Stable-Baselines' callables of the remaining fraction."""
    frac = 1.0 - u / spec["updates"]
    return 3e-4 * frac, 0.2 * frac + 0.05, 0.1 * frac


def trajectory(spec, world):
    """One seeded host-env trajectory of every global env (Discrete cases): reset observations and, per update, [T, N, O]."""
    rng = np.random.default_rng(7)
    N, T, O, U = spec["n_envs"] * world, spec["n_steps"], spec.get("obs_dim", 18), spec["updates"]
    obs0 = (rng.standard_normal((N, O)) * 2 + 0.5).astype(np.float32)
    raw = (rng.standard_normal((U, T, N, O)) * 2 + 0.5).astype(np.float32)
    rew = rng.standard_normal((U, T, N)).astype(np.float32)
    done = (rng.uniform(size=(U, T, N)) < 0.05).astype(np.float32)
    return obs0, raw, rew, done


def make_core(spec, rank, world, device):
    h1, h2 = spec["hidden"]
    return core.PPOCore(activation=spec.get("activation", "tanh"), action_space=spec.get("space", "box"), device=device,
                        obs_dim=spec.get("obs_dim", 18), act_dim=spec.get("act_dim", 18), hidden1=h1, hidden2=h2,
                        n_envs=spec["n_envs"], n_steps=spec["n_steps"], nminibatches=spec["nmb"], noptepochs=spec["epochs"],
                        ent_coef=ENT, seed=99, rank=rank, world_size=world, env_offset=rank * spec["n_envs"],
                        n_envs_global=spec["n_envs"] * world)


def run_case(name, spec, rank, world, device):
    out = {}
    c = make_core(spec, rank, world, device)
    c.init_orthogonal(5)
    setup_comm(core, c, rank, world)
    if world > 1:
        c.comm_set_p2p(spec.get("p2p", True))
    if spec.get("vf"):
        c.vf_clip = spec["vf"]
    c.shuffle_seed(SHUFFLE_SEED)
    discrete = spec.get("space") == "discrete"
    Nl = spec["n_envs"]
    mine = slice(rank * Nl, (rank + 1) * Nl)
    if discrete:
        obs0, raw, rew, done = trajectory(spec, world)
        c.runner_reset(obs0[mine])
        if rank == 0:
            out.update(traj_obs0=obs0, traj_raw=raw, traj_rew=rew, traj_done=done)
    else:
        c.synth_env_reset()
    out["p0"] = c.get_tensor("params")
    builds = []
    for u in range(spec["updates"]):
        lr, cr, cr_vf = schedule(spec, u)
        if discrete:
            c.runner_rollout_replay(raw[u][:, mine], rew[u][:, mine], done[u][:, mine])
        else:
            c.rollout_synthetic()
        for b in BUFS:
            out[f"u{u}_{b}"] = c.rollout_get(b)
        if u == 0:
            out.update({f"stats0_{k}": v for k, v in c.vecnorm_stats().items()})
        out[f"u{u}_losses"] = c.train_update(lr, cr, cliprange_vf=cr_vf if spec.get("vf") == "separate" else None)
        out[f"u{u}_perms"] = np.stack([c.train_get_permutation(e) for e in range(spec["epochs"])])
        out[f"u{u}_schedule"] = np.array([lr, cr, cr_vf])
        after, ks = spec.get("minibatches_after", (None, ()))
        if u == after:  # an even number of steps: the beta-power slot the update graph was captured with comes back
            out[f"u{u}_mb_ks"] = np.array(ks)
            out[f"u{u}_mb_losses"] = np.stack([c.train_minibatch(k, lr, cr)[0] for k in ks])
        builds.append(c.graph_builds())
    for t in ("params", "adam_m", "adam_v", "beta1_power", "beta2_power"):
        out[t] = c.get_tensor(t)
    out.update({f"stats_{k}": v for k, v in c.vecnorm_stats().items()})
    d = c.desc
    out.update(builds=np.array(builds), comm_error=np.array(c.comm_error()), family_train=np.array(c.kernel_family("train")),
               family_rollout=np.array(c.kernel_family("rollout")),
               hparams=np.array([d.ent_coef, d.vf_coef, d.max_grad_norm, d.adam_beta1, d.adam_beta2, d.adam_epsilon]))
    dist.barrier()  # no rank unmaps a mailbox a peer may still write to
    c.close()
    if rank == 0 and name in SINGLE_GPU_ROLLOUT:  # the global configuration on one GPU, first rollout
        g = make_core(dict(spec, n_envs=Nl * world), 0, 1, device)
        g.init_orthogonal(5)
        if spec.get("vf"):
            g.vf_clip = spec["vf"]
        g.synth_env_reset()
        g.rollout_synthetic()
        for b in BUFS:
            out[f"single_{b}"] = g.rollout_get(b)
        out.update({f"single_stats_{k}": v for k, v in g.vecnorm_stats().items()})
        g.close()
    return out


def main():
    out_dir = sys.argv[1]
    rank, world, local = env_world()
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cases = {**CASES, **PERM_CASES}
    for name, spec in cases.items():
        if world == 1 and spec.get("p2p") is False:
            continue  # one rank has nothing to exchange
        env = spec.get("env", ())
        for e in env:
            os.environ[e] = "1"
        try:
            out = run_case(name, spec, rank, world, local)
        finally:
            for e in env:
                del os.environ[e]
        np.savez(os.path.join(out_dir, f"{name}_r{rank}.npz"), **out)
        dist.barrier()
        if rank == 0:
            print(f"case {name}: done", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
