"""Per-update cost of a learning-rate / clip-range schedule: constant lr and cliprange against Stable-Baselines' linear
annealing (frac = 1 - (update - 1) / n_updates, new values every update), at C3, the C4 shard and c1x4096.

Two builds are compared in one call, alternating between them run by run: this tree and another checkout (--other, e.g.
the parent commit with its library built), each imported from its own tree in a fresh process.  Every run reports the
mean time of the train phase (ppo_train_update, host clock around a call that ends in a device synchronise) and of the
whole update, and how many CUDA graphs the core captured and instantiated (where the build can tell).  The card's name
and power limit are read in the same call.

    python tools/schedule_bench.py --other /path/to/parent --out profiles/schedule_bench.json
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
}


def worker(workload, schedule, updates, warmup):
    """Runs inside the tree on sys.path[0]: warm-up updates, then `updates` timed ones."""
    from ppo_cpp_b200 import core
    n_envs, n_steps, h1, h2, nmb, epochs = WORKLOADS[workload]
    c = core.PPOCore(hidden1=h1, hidden2=h2, n_envs=n_envs, n_steps=n_steps, nminibatches=nmb, noptepochs=epochs, seed=1234)
    c.init_orthogonal(7)
    c.shuffle_seed(5)
    c.synth_env_reset()
    total = warmup + updates
    builds = getattr(c, "graph_builds", None)
    train_ms, update_ms, losses = [], [], None
    for u in range(1, total + 1):
        frac = 1.0 - (u - 1) / total
        lr, cr = (2.5e-4 * frac, 0.2 * frac) if schedule == "annealed" else (2.5e-4, 0.2)
        t0 = time.perf_counter()
        c.rollout_synthetic()
        c.sync()
        t1 = time.perf_counter()
        losses = c.train_update(lr, cr)  # returns after the losses reached the host
        t2 = time.perf_counter()
        if u > warmup:
            train_ms.append(1e3 * (t2 - t1))
            update_ms.append(1e3 * (t2 - t0))
    out = {"train_ms": statistics.mean(train_ms), "train_ms_median": statistics.median(train_ms), "update_ms": statistics.mean(update_ms),
           "graph_builds": builds() if builds else None, "last_losses": [float(x) for x in losses]}
    c.close()
    return out


def run_in(tree, workload, schedule, updates, warmup):
    env = dict(os.environ, PYTHONPATH=tree)
    env.pop("PPO_CORE_LIB", None)  # each tree loads its own library
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", workload, schedule, str(updates), str(warmup)],
                       cwd=tree, env=env, capture_output=True, text=True, timeout=1800)
    if r.returncode != 0:
        raise RuntimeError(f"{tree} {workload} {schedule}: {r.stderr[-2000:]}")
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
    ap.add_argument("--worker", nargs=4, metavar=("WORKLOAD", "SCHEDULE", "UPDATES", "WARMUP"))
    ap.add_argument("--other", help="another checkout with its library built (e.g. the parent commit)")
    ap.add_argument("--workloads", default="c3,c4_shard,c1x4096")
    ap.add_argument("--updates", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=2, help="alternations of the two builds per (workload, schedule)")
    ap.add_argument("--out")
    args = ap.parse_args()
    if args.worker:
        w, s, n, k = args.worker
        print(json.dumps(worker(w, s, int(n), int(k))), flush=True)
        return
    trees = {"this": HERE}
    if args.other:
        trees["other"] = os.path.abspath(args.other)
    result = {"gpu": gpu_info(), "updates": args.updates, "warmup": args.warmup,
              "timing": "host clock; train = ppo_train_update incl. the losses' copy to the host; update = synthetic rollout + train",
              "runs": []}
    for wl in args.workloads.split(","):
        for sched in ("constant", "annealed"):
            for rep in range(args.reps):
                for name, tree in trees.items():
                    r = run_in(tree, wl, sched, args.updates, args.warmup)
                    r.update(build=name, workload=wl, schedule=sched, rep=rep)
                    result["runs"].append(r)
                    print(json.dumps(r), flush=True)
    summary = {}
    for r in result["runs"]:
        summary.setdefault(f'{r["workload"]} {r["schedule"]} {r["build"]}', []).append(r["train_ms"])
    result["summary_train_ms"] = {k: {"mean": statistics.mean(v), "runs": v} for k, v in summary.items()}
    print(json.dumps(result["summary_train_ms"], indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
