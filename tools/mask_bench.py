"""Cost of invalid-action masks: Discrete(12) and MultiDiscrete([4, 4, 4]), obs 18, [64,64], each head with masking off and on, for
the train phase of one update, the policy step on 4096 envs and one env step of the host-env protocol.

4096 envs x 64 steps, 32 minibatches, 10 epochs (C3's update); every arm runs the F family.  Every arm fills its rollout buffers through
the per-step host-env protocol (ppo_runner_act / ppo_runner_observe[_masked]) from the same recorded trajectory; the masked arms feed
random masks (about half the logits allowed, at least one per categorical), so each trains on its own policy's actions.

The four arms alternate run by run, each run in a fresh process.  train = ppo_train_update (host clock; the call returns after the
losses reached the host).  policy_step = ppo_policy_step / ppo_policy_step_masked on device pointers (PPO_DEVICE), CUDA events on the
core's stream over 200 back-to-back calls; the masked call includes packing the [4096, 12] byte mask into words.  The card's name and
power limit are read in the same call.  host_env_step = one ppo_runner_act (actions to host memory) + ppo_runner_observe[_masked] (host
observation, reward, done and, masked, the [4096, A] byte mask), host clock over the rollout's 64 steps up to its ppo_runner_finish
and a synchronise, the mean over the timed updates.

    python tools/mask_bench.py --out profiles/mask_bench.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
O, H1, H2 = 18, 64, 64
HEADS = {  # name: PPOCore keywords of the head, both over 12 logits
    "discrete_12": dict(action_space="discrete", act_dim=12),
    "multi_discrete_4_4_4": dict(action_space="multi_discrete", nvec=[4, 4, 4]),
}
ARMS = [(h, m) for h in HEADS for m in (False, True)]
N_ENVS, N_STEPS, NMB, EPOCHS = 4096, 64, 32, 10


def rand_masks(rng, slices, n):
    m = (rng.uniform(size=(n, slices[-1][1])) < 0.5).astype("uint8")
    for a, b in slices:
        empty = m[:, a:b].sum(1) == 0
        m[empty, a + rng.integers(0, b - a, int(empty.sum()))] = 1
    return m


def worker(head, masked, updates, warmup):
    """Runs inside the tree on sys.path[0]: warm-up updates, then `updates` timed ones."""
    import numpy as np
    import torch
    from ppo_cpp_b200 import core, _lib
    c = core.PPOCore(obs_dim=O, hidden1=H1, hidden2=H2, n_envs=N_ENVS, n_steps=N_STEPS, nminibatches=NMB, noptepochs=EPOCHS,
                     seed=1234, **HEADS[head])
    c.action_masking = masked
    c.init_orthogonal(7)
    c.shuffle_seed(5)
    nv = c.nvec if head != "discrete_12" else [12]
    off = np.concatenate([[0], np.cumsum(nv)])
    slices = [(int(off[i]), int(off[i + 1])) for i in range(len(nv))]
    rng = np.random.default_rng(3)
    raw = rng.standard_normal((N_STEPS, N_ENVS, O)).astype(np.float32)
    rew = rng.standard_normal((N_STEPS, N_ENVS)).astype(np.float32)
    done = (rng.uniform(size=(N_STEPS, N_ENVS)) < 0.01).astype(np.float32)
    masks = [rand_masks(rng, slices, N_ENVS) for _ in range(N_STEPS)] if masked else [None] * N_STEPS
    c.runner_reset(raw[0], mask=masks[-1])
    train_ms, step_us, losses = [], [], None
    for u in range(1, warmup + updates + 1):
        r0 = time.perf_counter()
        for t in range(N_STEPS):
            c.runner_act(t)
            c.runner_observe(t, raw[t], rew[t], done[t], mask=masks[t])
        c.runner_finish()
        c.sync()
        if u > warmup:
            step_us.append(1e6 * (time.perf_counter() - r0) / N_STEPS)
        t0 = time.perf_counter()
        losses = c.train_update(2.5e-4, 0.2)
        t1 = time.perf_counter()
        if u > warmup:
            train_ms.append(1e3 * (t1 - t0))
    # policy step on device pointers, CUDA events on the core's stream
    dev = torch.device("cuda", 0)
    obs = torch.tensor(raw[0], device=dev)
    mask = torch.tensor(masks[0], device=dev) if masked else None
    act = torch.zeros((N_ENVS, c.AW), device=dev)
    val = torch.zeros(N_ENVS, device=dev)
    nlp = torch.zeros(N_ENVS, device=dev)
    s = torch.cuda.ExternalStream(c.stream, device=dev)

    def step():
        if masked:
            r = c.lib.ppo_policy_step_masked(c._h, obs.data_ptr(), N_ENVS, None, mask.data_ptr(), act.data_ptr(), val.data_ptr(), nlp.data_ptr(), _lib.PPO_DEVICE)
        else:
            r = c.lib.ppo_policy_step(c._h, obs.data_ptr(), N_ENVS, None, act.data_ptr(), val.data_ptr(), nlp.data_ptr(), _lib.PPO_DEVICE)
        assert r == 0, c.lib.ppo_last_error()

    torch.cuda.synchronize()
    for _ in range(20):
        step()
    policy_ms = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(200):
            step()
        e1.record(s)
        e1.synchronize()
        policy_ms.append(e0.elapsed_time(e1) / 200)
    c.sync()
    out = {"train_ms": statistics.mean(train_ms), "train_ms_median": statistics.median(train_ms),
           "train_ms_stdev": statistics.stdev(train_ms) if len(train_ms) > 1 else 0.0,
           "policy_step_ms": statistics.median(policy_ms), "host_env_step_us": statistics.mean(step_us), "train_family": c.kernel_family("train"),
           "policy_family": c.kernel_family("policy"), "last_losses": [float(x) for x in losses]}
    c.close()
    return out


def run(head, masked, updates, warmup):
    env = dict(os.environ, PYTHONPATH=HERE)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", head, str(int(masked)), str(updates), str(warmup)],
                       cwd=HERE, env=env, capture_output=True, text=True, timeout=1800)
    if r.returncode != 0:
        raise RuntimeError(f"{head} masked={masked}: {r.stderr[-2000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60, check=True).stdout.strip().splitlines()
    return q[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", nargs=4, metavar=("HEAD", "MASKED", "UPDATES", "WARMUP"))
    ap.add_argument("--updates", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2, help="alternations of the four arms")
    ap.add_argument("--out")
    args = ap.parse_args()
    if args.worker:
        h, m, n, k = args.worker
        print(json.dumps(worker(h, bool(int(m)), int(n), int(k))), flush=True)
        return
    result = {"gpu": gpu_info(), "updates": args.updates, "warmup": args.warmup,
              "config": {"obs_dim": O, "hidden": [H1, H2], "n_envs": N_ENVS, "n_steps": N_STEPS, "nminibatches": NMB, "noptepochs": EPOCHS},
              "timing": "train = ppo_train_update, host clock, incl. the losses' copy to the host; policy_step = one ppo_policy_step[_masked] "
                        "call on device pointers, CUDA events over 200 calls, median of 3; host_env_step = ppo_runner_act + "
                        "ppo_runner_observe[_masked] with host buffers, host clock over a rollout of 64 steps up to its finish and a synchronise",
              "runs": []}
    for rep in range(args.reps):
        for head, masked in ARMS:
            r = run(head, masked, args.updates, args.warmup)
            r.update(head=head, masked=masked, rep=rep)
            result["runs"].append(r)
            print(json.dumps(r), flush=True)
    summary = {}
    for r in result["runs"]:
        s = summary.setdefault(f"{r['head']}/{'masked' if r['masked'] else 'unmasked'}",
                               {"train_ms": [], "policy_step_ms": [], "host_env_step_us": [], "train_family": r["train_family"]})
        for k in ("train_ms", "policy_step_ms", "host_env_step_us"):
            s[k].append(r[k])
    result["summary"] = {k: {"train_ms_mean": statistics.mean(v["train_ms"]), "policy_step_ms_mean": statistics.mean(v["policy_step_ms"]),
                             "host_env_step_us_mean": statistics.mean(v["host_env_step_us"]), **v}
                         for k, v in summary.items()}
    for h in HEADS:
        a, b = result["summary"][f"{h}/unmasked"], result["summary"][f"{h}/masked"]
        result["summary"][f"{h}/overhead"] = {"train": b["train_ms_mean"] / a["train_ms_mean"] - 1.0,
                                              "policy_step": b["policy_step_ms_mean"] / a["policy_step_ms_mean"] - 1.0,
                                              "host_env_step": b["host_env_step_us_mean"] / a["host_env_step_us_mean"] - 1.0}
    print(json.dumps(result["summary"], indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
