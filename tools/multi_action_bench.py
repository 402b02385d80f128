"""Cost of the MultiDiscrete and MultiBinary policy heads against the categorical head over the same 12 logits: Discrete(12),
MultiDiscrete([4, 4, 4]) and MultiBinary(12), obs 18, [64,64], for the train phase of one update and for the policy step.

4096 envs x 64 steps, 32 minibatches, 10 epochs (C3's update); every head runs the F family.  Each core fills its rollout
buffers from the same recorded host trajectory (ppo_runner_rollout_replay), so each trains on its own policy's actions.

The three heads alternate run by run, each run in a fresh process.  train = ppo_train_update (host clock; the call returns
after the losses reached the host), policy = ppo_profile_kernel("policy_step") (CUDA events over back-to-back launches on
4096 envs).  The card's name and power limit are read in the same call.

    python tools/multi_action_bench.py --out profiles/multi_action_bench.json
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
HEADS = {  # name: PPOCore keywords of the head, all over 12 logits
    "discrete_12": dict(action_space="discrete", act_dim=12),
    "multi_discrete_4_4_4": dict(action_space="multi_discrete", nvec=[4, 4, 4]),
    "multi_binary_12": dict(action_space="multi_binary", act_dim=12),
}
N_ENVS, N_STEPS, NMB, EPOCHS = 4096, 64, 32, 10


def worker(head, updates, warmup):
    """Runs inside the tree on sys.path[0]: warm-up updates, then `updates` timed ones."""
    import numpy as np
    from ppo_cpp_b200 import core
    c = core.PPOCore(obs_dim=O, hidden1=H1, hidden2=H2, n_envs=N_ENVS, n_steps=N_STEPS, nminibatches=NMB, noptepochs=EPOCHS,
                     seed=1234, **HEADS[head])
    c.init_orthogonal(7)
    c.shuffle_seed(5)
    rng = np.random.default_rng(3)
    raw = rng.standard_normal((N_STEPS, N_ENVS, O)).astype(np.float32)
    rew = rng.standard_normal((N_STEPS, N_ENVS)).astype(np.float32)
    done = (rng.uniform(size=(N_STEPS, N_ENVS)) < 0.01).astype(np.float32)
    c.runner_reset(raw[0])
    train_ms, losses = [], None
    for u in range(1, warmup + updates + 1):
        c.runner_rollout_replay(raw, rew, done)
        c.sync()
        t0 = time.perf_counter()
        losses = c.train_update(2.5e-4, 0.2)
        t1 = time.perf_counter()
        if u > warmup:
            train_ms.append(1e3 * (t1 - t0))
    policy_ms = [c.profile_kernel("policy_step", 200) for _ in range(3)]
    out = {"train_ms": statistics.mean(train_ms), "train_ms_median": statistics.median(train_ms),
           "train_ms_stdev": statistics.stdev(train_ms) if len(train_ms) > 1 else 0.0,
           "policy_step_ms": statistics.median(policy_ms), "train_family": c.kernel_family("train"),
           "policy_family": c.kernel_family("policy"), "last_losses": [float(x) for x in losses]}
    c.close()
    return out


def run(head, updates, warmup):
    env = dict(os.environ, PYTHONPATH=HERE)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", head, str(updates), str(warmup)],
                       cwd=HERE, env=env, capture_output=True, text=True, timeout=1800)
    if r.returncode != 0:
        raise RuntimeError(f"{head}: {r.stderr[-2000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60, check=True).stdout.strip().splitlines()
    return q[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", nargs=3, metavar=("HEAD", "UPDATES", "WARMUP"))
    ap.add_argument("--updates", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2, help="alternations of the three heads")
    ap.add_argument("--out")
    args = ap.parse_args()
    if args.worker:
        h, n, k = args.worker
        print(json.dumps(worker(h, int(n), int(k))), flush=True)
        return
    result = {"gpu": gpu_info(), "updates": args.updates, "warmup": args.warmup,
              "config": {"obs_dim": O, "hidden": [H1, H2], "n_envs": N_ENVS, "n_steps": N_STEPS, "nminibatches": NMB, "noptepochs": EPOCHS},
              "timing": "train = ppo_train_update, host clock, incl. the losses' copy to the host; "
                        "policy_step = ppo_profile_kernel('policy_step', 200), CUDA events, median of 3",
              "runs": []}
    for rep in range(args.reps):
        for head in HEADS:
            r = run(head, args.updates, args.warmup)
            r.update(head=head, rep=rep)
            result["runs"].append(r)
            print(json.dumps(r), flush=True)
    summary = {}
    for r in result["runs"]:
        s = summary.setdefault(r["head"], {"train_ms": [], "policy_step_ms": [], "train_family": r["train_family"]})
        s["train_ms"].append(r["train_ms"])
        s["policy_step_ms"].append(r["policy_step_ms"])
    result["summary"] = {k: {"train_ms_mean": statistics.mean(v["train_ms"]), "policy_step_ms_mean": statistics.mean(v["policy_step_ms"]), **v}
                         for k, v in summary.items()}
    print(json.dumps(result["summary"], indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
