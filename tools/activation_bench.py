"""Per-update cost of the hidden-layer activation: tanh against ReLU cores built from the same seed, at C3 (U train family
+ R rollout), the C4 shard (W), c1x4096 (S) and C1 (the S epoch kernel + the single-env rollout walk).

The two activations alternate run by run, each run in a fresh process.  Every run reports the mean time of the rollout
(ppo_rollout_synthetic) and of the train phase (ppo_train_update), host clock around calls that end in a device
synchronise, and the losses of its last update.  The card's name and power limit are read in the same call.

    python tools/activation_bench.py --out profiles/activation_bench.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = {  # name: (n_envs, n_steps, h1, h2, nminibatches, noptepochs) as in bench.py
    "c3": (4096, 64, 64, 64, 32, 10),
    "c4_shard": (8192, 64, 256, 256, 32, 10),
    "c1x4096": (4096, 64, 4, 5, 32, 10),
    "c1": (1, 2048, 4, 5, 32, 10),
}


def worker(workload, activation, updates, warmup):
    """Runs inside the tree on sys.path[0]: warm-up updates, then `updates` timed ones."""
    from ppo_cpp_b200 import core
    n_envs, n_steps, h1, h2, nmb, epochs = WORKLOADS[workload]
    c = core.PPOCore(activation=activation, hidden1=h1, hidden2=h2, n_envs=n_envs, n_steps=n_steps, nminibatches=nmb, noptepochs=epochs, seed=1234)
    c.init_orthogonal(7)
    c.shuffle_seed(5)
    c.synth_env_reset()
    total = warmup + updates
    train_ms, rollout_ms, losses = [], [], None
    for u in range(1, total + 1):
        c.sync()
        t0 = time.perf_counter()
        c.rollout_synthetic()
        c.sync()
        t1 = time.perf_counter()
        losses = c.train_update(2.5e-4, 0.2)  # returns after the losses reached the host
        t2 = time.perf_counter()
        if u > warmup:
            train_ms.append(1e3 * (t2 - t1))
            rollout_ms.append(1e3 * (t1 - t0))
    out = {"train_ms": statistics.mean(train_ms), "train_ms_median": statistics.median(train_ms), "rollout_ms": statistics.mean(rollout_ms),
           "rollout_ms_median": statistics.median(rollout_ms), "train_family": c.kernel_family("train"),
           "rollout_family": c.kernel_family("rollout"), "last_losses": [float(x) for x in losses]}
    c.close()
    return out


def run(workload, activation, updates, warmup):
    env = dict(os.environ, PYTHONPATH=HERE)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", workload, activation, str(updates), str(warmup)],
                       cwd=HERE, env=env, capture_output=True, text=True, timeout=1800)
    if r.returncode != 0:
        raise RuntimeError(f"{workload} {activation}: {r.stderr[-2000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except OSError:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", nargs=4, metavar=("WORKLOAD", "ACTIVATION", "UPDATES", "WARMUP"))
    ap.add_argument("--workloads", default="c3,c4_shard,c1x4096,c1")
    ap.add_argument("--updates", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=2, help="alternations of the two activations per workload")
    ap.add_argument("--out")
    args = ap.parse_args()
    if args.worker:
        w, s, n, k = args.worker
        print(json.dumps(worker(w, s, int(n), int(k))), flush=True)
        return
    result = {"gpu": gpu_info(), "updates": args.updates, "warmup": args.warmup,
              "timing": "host clock; train = ppo_train_update incl. the losses' copy to the host; rollout = ppo_rollout_synthetic",
              "runs": []}
    for wl in args.workloads.split(","):
        for rep in range(args.reps):
            for act in ("tanh", "relu"):
                r = run(wl, act, args.updates, args.warmup)
                r.update(workload=wl, activation=act, rep=rep)
                result["runs"].append(r)
                print(json.dumps(r), flush=True)
    summary = {}
    for r in result["runs"]:
        s = summary.setdefault(f'{r["workload"]} {r["activation"]}', {"train_ms": [], "rollout_ms": []})
        s["train_ms"].append(r["train_ms"])
        s["rollout_ms"].append(r["rollout_ms"])
    result["summary"] = {k: {"train_ms_mean": statistics.mean(v["train_ms"]), "rollout_ms_mean": statistics.mean(v["rollout_ms"]), **v}
                         for k, v in summary.items()}
    print(json.dumps(result["summary"], indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
