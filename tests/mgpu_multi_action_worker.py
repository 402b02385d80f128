"""Worker of test_multi_action.py's sharded updates: one process per GPU under torch.distributed.run,
    python -m torch.distributed.run --nnodes 1 --nproc-per-node W --master-addr 127.0.0.1 --master-port P \\
        tests/mgpu_multi_action_worker.py OUT_DIR
Runs every case of CASES (the MultiDiscrete and MultiBinary heads on the F and T families, and over the NCCL fallback) on
sharded cores fed from one recorded host-env trajectory of all global envs, and writes what each rank holds to
OUT_DIR/<case>_r<rank>.npz: its own rollout rows of every update, the permutations, losses, params, Adam state and kernel family.
It computes no reference and asserts nothing; the test does both."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppo_cpp_b200 import core  # noqa: E402
from ppo_cpp_b200.dist import env_world, setup_comm  # noqa: E402
from mgpu_parity_worker import BUFS, ENT, SHUFFLE_SEED, schedule, trajectory  # noqa: E402

O, NVEC, NB = 6, [3, 5, 2], 6  # the shapes of test_multi_action.py's fp64 reference
HEADS = {"md": dict(action_space="multi_discrete", nvec=NVEC), "mb": dict(action_space="multi_binary", act_dim=NB)}
# per-rank sizes; the global run is W times as many envs
_BASE = dict(hidden=(64, 64), obs_dim=O, n_envs=128, n_steps=16, nmb=4, epochs=2, updates=2)
CASES = {}
for _h in HEADS:
    CASES[f"{_h}_fused"] = dict(_BASE, head=_h)
    CASES[f"{_h}_tile"] = dict(_BASE, head=_h, activation="relu", env=("PPO_DISABLE_FUSED",))
    CASES[f"{_h}_nccl"] = dict(_BASE, head=_h, p2p=False)  # gradients by ncclAllReduce, no graphs


def make_core(spec, rank, world, device):
    h1, h2 = spec["hidden"]
    return core.PPOCore(activation=spec.get("activation", "tanh"), device=device, obs_dim=O, hidden1=h1, hidden2=h2,
                        n_envs=spec["n_envs"], n_steps=spec["n_steps"], nminibatches=spec["nmb"], noptepochs=spec["epochs"],
                        ent_coef=ENT, seed=99, rank=rank, world_size=world, env_offset=rank * spec["n_envs"],
                        n_envs_global=spec["n_envs"] * world, **HEADS[spec["head"]])


def run_case(spec, rank, world, device):
    out = {}
    c = make_core(spec, rank, world, device)
    c.init_orthogonal(5)
    setup_comm(core, c, rank, world)
    if world > 1:
        c.comm_set_p2p(spec.get("p2p", True))
    c.shuffle_seed(SHUFFLE_SEED)
    Nl = spec["n_envs"]
    mine = slice(rank * Nl, (rank + 1) * Nl)
    obs0, raw, rew, done = trajectory(spec, world)
    c.runner_reset(obs0[mine])
    out["p0"] = c.get_tensor("params")
    for u in range(spec["updates"]):
        lr, cr, _ = schedule(spec, u)
        c.runner_rollout_replay(raw[u][:, mine], rew[u][:, mine], done[u][:, mine])
        for b in BUFS:
            out[f"u{u}_{b}"] = c.rollout_get(b)
        out[f"u{u}_losses"] = c.train_update(lr, cr)
        out[f"u{u}_perms"] = np.stack([c.train_get_permutation(e) for e in range(spec["epochs"])])
        out[f"u{u}_schedule"] = np.array([lr, cr])
    for t in ("params", "adam_m", "adam_v", "beta1_power", "beta2_power"):
        out[t] = c.get_tensor(t)
    d = c.desc
    out.update(comm_error=np.array(c.comm_error()), family_train=np.array(c.kernel_family("train")),
               hparams=np.array([d.ent_coef, d.vf_coef, d.max_grad_norm, d.adam_beta1, d.adam_beta2, d.adam_epsilon]))
    dist.barrier()  # no rank unmaps a mailbox a peer may still write to
    c.close()
    return out


def main():
    out_dir = sys.argv[1]
    rank, world, local = env_world()
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    for name, spec in CASES.items():
        if world == 1 and spec.get("p2p") is False:
            continue  # one rank has nothing to exchange
        env = spec.get("env", ())
        for e in env:
            os.environ[e] = "1"
        try:
            out = run_case(spec, rank, world, local)
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
