"""Worker of test_action_masks.py's sharded masked updates: one process per GPU under torch.distributed.run,
    python -m torch.distributed.run --nnodes 1 --nproc-per-node W --master-addr 127.0.0.1 --master-port P \\
        tests/mgpu_action_mask_worker.py OUT_DIR
Runs every case of CASES (the Discrete and MultiDiscrete heads with action masks on the F and T families, and over the NCCL
fallback) on sharded masking cores.  Every rank steps its share of one seeded trajectory of all global envs through the host-env
protocol with that trajectory's masks (ppo_runner_reset_masked / act / observe_masked), and writes what it holds to
OUT_DIR/<case>_r<rank>.npz: its own rollout rows of every update (the masks among them), the masks it fed, the permutations,
losses, params, Adam state and kernel family.  It computes no reference and asserts nothing; the test does both."""
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

O, N_DISC, NVEC = 6, 7, [3, 5, 2]  # the shapes of test_action_masks.py's fp64 reference
HEADS = {"disc": dict(action_space="discrete", act_dim=N_DISC), "md": dict(action_space="multi_discrete", nvec=NVEC)}
SLICES = {"disc": [(0, N_DISC)], "md": [(0, 3), (3, 8), (8, 10)]}
# per-rank sizes; the global run is W times as many envs
_BASE = dict(hidden=(64, 64), obs_dim=O, n_envs=128, n_steps=16, nmb=4, epochs=2, updates=2)
CASES = {}
for _h in HEADS:
    CASES[f"{_h}_fused"] = dict(_BASE, head=_h)
    CASES[f"{_h}_tile"] = dict(_BASE, head=_h, activation="relu", env=("PPO_DISABLE_FUSED",))
    CASES[f"{_h}_nccl"] = dict(_BASE, head=_h, p2p=False)  # gradients by ncclAllReduce, no graphs


def mask_trajectory(spec, world):
    """Seeded masks of every global env: [U, T + 1, N, A] (index 0 of update 0: the reset's), about half the logits allowed, at
    least one per slice."""
    rng = np.random.default_rng(11)
    N, T, U, sl = spec["n_envs"] * world, spec["n_steps"], spec["updates"], SLICES[spec["head"]]
    m = (rng.uniform(size=(U, T + 1, N, sl[-1][1])) < 0.5).astype(np.uint8)
    for a, b in sl:
        empty = m[..., a:b].sum(-1) == 0
        m[..., a][empty] = 1
    return m


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
    c.action_masking = True
    setup_comm(core, c, rank, world)
    if world > 1:
        c.comm_set_p2p(spec.get("p2p", True))
    c.shuffle_seed(SHUFFLE_SEED)
    Nl, T = spec["n_envs"], spec["n_steps"]
    mine = slice(rank * Nl, (rank + 1) * Nl)
    obs0, raw, rew, done = trajectory(spec, world)
    masks = mask_trajectory(spec, world)[:, :, mine]
    c.runner_reset(obs0[mine], mask=masks[0, 0])
    cur = masks[0, 0]
    out["p0"] = c.get_tensor("params")
    for u in range(spec["updates"]):
        lr, cr, _ = schedule(spec, u)
        fed = []
        for t in range(T):
            c.runner_act(t)
            fed.append(cur)
            cur = masks[u, t + 1]
            c.runner_observe(t, raw[u][t, mine], rew[u][t, mine], done[u][t, mine], mask=cur)
        c.runner_finish()
        for b in BUFS + ("action_masks",):
            out[f"u{u}_{b}"] = c.rollout_get(b)
        out[f"u{u}_fed_masks"] = np.stack(fed)  # [T, Nl, A]: the mask in force at each step
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
