#!/usr/bin/env python
"""Benchmark of the PPO hot path (BASELINE.json metric: PPO env-steps/s and update samples/s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c1|c4] [--dump-outputs DIR]

A "step" is one PPO update: rollout of n_steps x n_envs transitions on the GPU-resident synthetic 18-dim env
(policy step + env + VecNormalize per env step, then GAE) followed by noptepochs x nminibatches train steps.
`value` = env-steps/s = n_batch / time(update), the reference's own fps formula (ppo2/ppo2.hpp:337-341).
Default workload = BASELINE.json configs[2] (C3): 4096 envs/GPU, MLP [64,64], n_steps 64 (262 144
transitions per update per GPU), 32 minibatches, 10 epochs.  Multi-GPU is weak scaling: every rank owns 4096
envs; per-minibatch gradients are allreduced with NCCL.

--impl reference times the CPU restatement of the reference (oracle/, OpenMP over all host cores) on the same
config — TensorFlow 1.14/Eigen are not installable, see DESIGN.md.

--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (see dump_outputs), so that two builds
can be compared output for output: every input is seeded, the same arguments give the same inputs.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree, which may be read-only

WORKLOADS = {
    # name: (n_envs per GPU, n_steps, h1, h2, nminibatches, noptepochs, description)
    "c3": (4096, 64, 64, 64, 32, 10, "C3: synthetic 18-dim env, 4096 envs/GPU, MLP [64,64], 262144 transitions/update/GPU"),
    "c1": (1, 2048, 4, 5, 32, 10, "C1 shape: 1 env, MLP [4,5], n_steps 2048 (reference CLI defaults)"),
    "c4": (8192, 64, 256, 256, 32, 10, "C4 shard: 8192 envs/GPU, MLP [256,256], 524288 transitions/update/GPU"),
    "c1x4096": (4096, 64, 4, 5, 32, 10, "reference net [4,5] on 4096 synthetic envs"),
    "c3x8": (32768, 64, 64, 64, 32, 10, "C3 net on 32768 envs (the global batch of an 8-GPU C3 run, on one GPU)"),
}
LR, CLIPRANGE = 3.9e-4, 0.161
METRIC, UNIT = "ppo_env_steps_per_sec", "env-steps/s"


def make_config(workload, world):
    """The `config` object of the JSON line — built by ONE function so that both arms print the same keys and values."""
    n_envs, n_steps, h1, h2, nmb, epochs, desc = WORKLOADS[workload]
    nbg = n_envs * n_steps * world
    return {"workload": desc, "n_envs_per_gpu": n_envs, "n_steps": n_steps, "hidden": [h1, h2], "nminibatches": nmb,
            "noptepochs": epochs, "global_batch": nbg, "minibatch": nbg // nmb, "parallelism": f"dp{world}",
            "l2": "256 MiB memset between timed steps (L2 flush), outside the per-step event pairs",
            "weights": "orthogonal random init (no graph file exists for this size)"}


def host_threads():
    """Host cores this process may use.  torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm must not inherit that."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def train_flops_per_sample(O, A, h1, h2):
    fwd = 2 * (O * h1 + h1 * h2) + h2 * A + h2
    dx = 2 * (h1 * h2) + h2 * A + h2
    return 2 * (2 * fwd + dx)


def cpu_learner(workload, threads=0):
    """The CPU restatement, structured like the reference (oracle/ppo_oracle.c oracle_learner_*)."""
    import ctypes as C

    import numpy as np

    import oracle_lib as ol
    n_envs, n_steps, h1, h2, nmb, epochs, _ = WORKLOADS[workload]
    lib = ol.load(fast=True)
    o = ol.Oracle(h1=h1, h2=h2, fast=True)
    rng = np.random.default_rng(0)
    params = (rng.standard_normal(o.Pq) * 0.1).astype(np.float32)
    params[o.offset(12):o.offset(13)] = 0.0
    return lib, o, params, (n_envs, n_steps, h1, h2, nmb, epochs)


def time_cpu_update(workload, epochs_run, reps=1, threads=0, world=1):
    """(seconds per full update extrapolated to all epochs, threads used, rollout s, per-epoch s).
    world > 1: the GLOBAL batch of a `world`-GPU run (n_envs x world envs), as one CPU job."""
    import ctypes as C

    import numpy as np

    import oracle_lib as ol
    threads = threads or host_threads()
    lib, o, params, (n_envs, n_steps, h1, h2, nmb, epochs) = cpu_learner(workload, threads)
    n_envs *= world
    d = ol.LearnerDesc(ol.Dims(18, 18, h1, h2), ol.HParams(0.0007160293171182275, 0.5, 0.5, 0.9, 0.999, 1e-5), n_envs, n_steps, nmb,
                       epochs_run, 0.99, 0.95, LR, CLIPRANGE, 1, 42, 0, threads)
    L = lib.oracle_learner_create(C.byref(d), params)
    used = lib.oracle_learner_threads(L)
    losses = np.zeros(5, np.float32)
    t_roll, t_train = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        lib.oracle_learner_rollout(L)
        t1 = time.perf_counter()
        lib.oracle_learner_train(L, losses)
        t2 = time.perf_counter()
        t_roll.append(t1 - t0)
        t_train.append((t2 - t1) / max(epochs_run, 1))
    lib.oracle_learner_destroy(L)
    r, e = min(t_roll), min(t_train)
    return r + epochs * e, used, r, e


def run_reference(args):
    """The reference's CPU implementation of the path (the oracle port: TF 1.14 / Eigen are not installable, DESIGN.md §5) on
    ALL host cores, on the same GLOBAL config as `--impl ours --gpus N` (N x 4096 envs), each step a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    world = max(1, args.gpus)
    n_envs, n_steps, h1, h2, nmb, epochs, desc = WORKLOADS[args.workload]
    n_batch = n_envs * n_steps * world
    threads = host_threads()
    os.environ["OMP_NUM_THREADS"] = str(threads)  # before libgomp initialises (torchrun set it to 1)
    # size the per-step sample so that (steps + warmup) steps end within a few minutes
    probe_total, threads, r, e = time_cpu_update(args.workload, 1, threads=threads, world=world)
    budget = 150.0 / max(args.steps + args.warmup, 1)
    epochs_run = max(1, min(epochs, int((budget - r) / max(e, 1e-9))))
    runs, spent = [], 0.0
    for i in range(args.steps + args.warmup):
        if runs and spent + (r + epochs_run * e) > 200.0:
            break  # bounded: never more than a few minutes in total
        total, threads, r, e = time_cpu_update(args.workload, epochs_run, threads=threads, world=world)
        spent += r + epochs_run * e
        runs.append(total)
    times = runs[args.warmup:] or runs[-1:]
    sec = statistics.mean(times) if times else probe_total
    value = n_batch / sec
    sample = (f"per step: full rollout ({n_steps} steps x {n_envs * world} envs) + {epochs_run} of {epochs} epochs of {nmb} minibatches, "
              f"train time scaled to {epochs} epochs; {len(times)} such steps timed")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": make_config(args.workload, world),
        "note": "CPU restatement of ppo_cpp (TensorFlow 1.14 / Eigen not installable); rank 0 runs the GLOBAL batch of the N-GPU config on all host cores",
        "update_samples_per_sec": n_batch / e,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples, time-stamped on arrival; `window()` summarises those
    that fell inside the timed region."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=20):
        self.rows, self.proc, self.index, self.period_ms = [], None, index, period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.period_ms)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def wait_first(self, timeout=8.0):
        t0 = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def window(self, t0, t1):
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 and len(r) >= 9]
        sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in rows if r[3].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


DUMP_MAX_ROWS = 262144  # all of C3's rollout; 168 B per transition over the eight buffers keeps a dump under 64 MB


def dump_outputs(core, c, out_dir):
    """What a caller of the timed path holds after its last update, one DIR/<name>.npy each: the weights and the Adam state
    (params, adam_m, adam_v, beta1_power, beta2_power), the VecNormalize statistics (vecnorm_*, counts in float64) and the
    rollout buffers of that update (rollout_*, rows as ppo_rollout_get lays them out).  Rollouts of more than DUMP_MAX_ROWS
    transitions are cut to the same seeded sample of rows in every run, whose indices go to rollout_rows.npy."""
    import numpy as np
    out = {name: c.get_tensor(name) for name in ("params", "adam_m", "adam_v", "beta1_power", "beta2_power")}
    for k, v in c.vecnorm_stats().items():
        out["vecnorm_" + k] = np.asarray(v, np.float64) if k.endswith("count") else v
    rows = None
    if c.n_batch > DUMP_MAX_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(c.n_batch, DUMP_MAX_ROWS, replace=False))
        out["rollout_rows"] = rows.astype(np.float64)
    for name in core.BUFFER_WIDTH:
        buf = c.rollout_get(name)
        out["rollout_" + name] = buf if rows is None else buf[rows]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from ppo_cpp_b200 import core

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE line (the JSON): whatever libraries print on the way (NCCL's version banner, ...) goes to stderr
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_envs, n_steps, h1, h2, nmb, epochs, desc = WORKLOADS[args.workload]
    n_batch_local = n_envs * n_steps
    n_batch_global = n_batch_local * world

    c = core.PPOCore(device=local, hidden1=h1, hidden2=h2, n_envs=n_envs, n_steps=n_steps, nminibatches=nmb, noptepochs=epochs,
                     seed=1234, rank=rank, world_size=world, env_offset=rank * n_envs, n_envs_global=n_envs * world)
    c.init_orthogonal(7)  # random-init weights of the named architecture, identical on every rank
    if world > 1:
        from ppo_cpp_b200.dist import setup_comm
        setup_comm(core, c, rank, world)  # NCCL communicator + peer mailboxes (NVLink P2P)
    c.shuffle_seed(42)
    c.synth_env_reset()
    stream = torch.cuda.ExternalStream(c.stream, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        c.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def one_update(ev0=None, ev1=None, evm=None):
        if ev0 is not None:
            ev0.record(stream)
        c.rollout_synthetic()
        if evm is not None:
            evm.record(stream)
        c.train_update(LR, CLIPRANGE, want_losses=False)
        if ev1 is not None:
            ev1.record(stream)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        one_update()
    barrier()
    if rank == 0:
        sampler.wait_first()
    c.counters(reset=True)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for e0, e1, em in evs:
        with torch.cuda.stream(stream):
            flush.zero_()  # L2 flush between timed steps, outside the timed interval
        one_update(e0, e1, em)
    barrier()
    t_wall1 = time.perf_counter()
    t_wall = t_wall1 - t_wall0
    ctr = c.counters()
    if rank == 0 and args.dump_outputs:
        dump_outputs(core, c, args.dump_outputs)  # before anything below moves the core's state on
    clocks = None
    if rank == 0:
        clocks = sampler.window(t_wall0, t_wall1)
        clocks["window"] = "timed region"
        if clocks["samples"] < 3 and world == 1:
            # timed region shorter than a few sampling periods: keep the same load running (untimed) until the
            # sampler has seen it, and say so
            t_x0 = time.perf_counter()
            while time.perf_counter() - t_x0 < 0.5:
                one_update()
                c.sync()
            clocks = sampler.window(t_wall0, time.perf_counter())
            clocks["window"] = "timed region + 0.5 s of the same load (timed region shorter than 3 sampling periods)"
        sampler.stop()
    if world > 1:
        dist.barrier()
    ms_total = sum(e0.elapsed_time(e1) for e0, e1, _ in evs)
    ms_train = sum(em.elapsed_time(e1) for _, e1, em in evs)
    t = torch.tensor([ms_total, ms_train], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_train = float(t[0]), float(t[1])
    ms_per_step = ms_total / args.steps
    value = n_batch_global / (ms_per_step * 1e-3)
    upd_sps = n_batch_global * epochs / (ms_train / args.steps * 1e-3)

    # ---- roofline of the dominant kernel (loss fwd + bwd), timed alone with CUDA events on the core's stream
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    k_ms = c.profile_kernel("train_fwdbwd", 64)
    family = c.kernel_family("train")
    per_rank_B = n_batch_global // nmb // world
    flops = per_rank_B * train_flops_per_sample(18, 18, h1, h2)
    bytes_alg = per_rank_B * 160
    tensor_peak = peaks.get("bf16_tflops", 1590.0)  # burst figure: the kernel is timed alone
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    ach_tf = flops / (k_ms * 1e-3) / 1e12
    ach_gb = bytes_alg / (k_ms * 1e-3) / 1e9
    on_tensor = "tcgen05" in family
    wide = min(h1, h2) >= 64
    src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
    if wide:  # dense-GEMM regime: algorithmic fp32 FLOPs against the measured bf16 tensor peak
        roofline = {"bound": "tensor", "achieved": ach_tf, "peak": tensor_peak, "unit": "TFLOP/s", "frac": ach_tf / tensor_peak,
                    "peak_source": src + " bf16_tflops (burst)",
                    "note": "fp32 parity costs 3 fp16 MMAs per fp32 MAC (fp16x2 split: hi*hi, hi*lo, lo*hi), so frac <= 1/3 on this pipe; the kernel is a latency chain (one 128-sample tile per CTA, 13 dependent GEMM -> epilogue phases), not a throughput problem: DESIGN.md 3.3" if on_tensor
                    else "runs on the fp32 FFMA pipe (nominal 74.4 TFLOP/s)"}
    else:  # tiny nets: 160 B per sample against the measured HBM copy bandwidth
        roofline = {"bound": "hbm", "achieved": ach_gb, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gb / hbm_peak,
                    "peak_source": src + " hbm_gbs"}
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f).get(args.workload)
        if tj and tj["kernel"].split("<")[0] in family:
            traffic = tj["bytes_per_launch"]
    except Exception:
        pass
    # the timed region itself: one epoch of the update = nmb minibatch steps (for the persistent U family ONE cooperative
    # launch that also holds the slab reduce, the gradient exchange, the norm clip and Adam); shuffle and advantage
    # statistics of the update are inside this time too
    epoch_ms = ms_train / args.steps / max(epochs, 1)
    roofline["in_timed_region"] = {"what": "train time of the timed region / epochs: %d minibatch steps incl. reduce + clip + Adam" % nmb,
                                   "epoch_ms": epoch_ms, "tflops": flops * nmb / (epoch_ms * 1e-3) / 1e12,
                                   "frac_of_fp32_ffma_nominal": flops * nmb / (epoch_ms * 1e-3) / 1e12 / 74.4}
    roofline.update({"kernel": family + ", one minibatch of %d samples per GPU, forward + backward alone" % per_rank_B, "traffic": traffic, "kernel_ms": k_ms,
                     "flops_per_launch": flops, "bytes_per_launch": bytes_alg, "tflops": ach_tf, "frac_of_fp32_ffma_nominal": ach_tf / 74.4,
                     "hbm_gbs": ach_gb})
    kernels = {}
    for name in ("policy_step", "norm_moments", "norm_apply", "gae", "grad_reduce", "adam"):
        try:
            kernels[name + "_ms"] = c.profile_kernel(name, 32)
        except Exception as ex:  # noqa: BLE001
            kernels[name + "_ms"] = str(ex)

    # ---- end to end through the C ABI with HOST buffers (Runner::run protocol against a host env)
    e2e = None
    if args.e2e:
        rng = np.random.default_rng(rank)
        pin = lambda shape: torch.empty(shape, dtype=torch.float32, pin_memory=True).numpy()  # noqa: E731
        raw_obs, raw_rew, raw_done, act = pin((n_steps, n_envs, 18)), pin((n_steps, n_envs)), pin((n_steps, n_envs)), pin((n_steps, n_envs, 18))
        raw_obs[:] = rng.standard_normal(raw_obs.shape)
        raw_rew[:] = rng.standard_normal(raw_rew.shape)
        raw_done[:] = rng.random(raw_done.shape) < 1 / 334
        losses = np.zeros(5, np.float32)

        def host_update():
            # the loop of Runner::run in C (ppo_runner_rollout_replay): per env step D2H of the actions for the host env,
            # H2D of what the host env returned (here: the next rows of the recorded arrays), then bootstrap + GAE
            c.runner_rollout_replay(raw_obs, raw_rew, raw_done, act)
            return c.train_update(LR, CLIPRANGE, want_losses=True)      # D2H: the update's mean losses

        c.runner_reset(raw_obs[0])
        host_update()
        barrier()
        c.counters(reset=True)
        k_e2e = max(1, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            losses = host_update()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ce = c.counters()
        e2e = {"value": n_batch_global * k_e2e / float(tt[0]), "unit": UNIT, "h2d_bytes_per_step": ce["h2d_bytes"] // k_e2e,
               "d2h_bytes_per_step": ce["d2h_bytes"] // k_e2e, "steps": k_e2e, "ms_per_step": float(tt[0]) / k_e2e * 1e3,
               "path": "ppo_runner_rollout_replay (Runner::run against a host env as one persistent kernel: per env step the actions are stored into the caller's pinned array over PCIe, the env's obs come back through the copy engine with a flag copy behind them, rewards / dones through mapped memory) + ppo_train_update with pinned HOST buffers, host env = replayed synthetic arrays",
               "final_losses": [float(x) for x in losses]}

    # ---- multi-GPU parity, outside the timed region: the run sharded over `world` ranks against ONE GPU running the same
    # global configuration (same Philox streams by global env id, same global permutation), and replica bit-identity
    parity = None
    if world > 1 and args.parity:
        parity = multi_gpu_parity(rank, world, local, (h1, h2))

    # ---- BASELINE.json configs[3] (C4): 65 536 envs, MLP [256,256] (W family, tcgen05 layer-wise GEMMs), 4 M transitions per
    # update sharded over the `world` GPUs — strong scaling: the global batch is fixed, every rank owns 65 536 / world envs
    c4 = None
    if world > 1 and args.c4 and 65536 % world == 0:
        c.close()
        c = None
        c4 = c4_sharded(core, rank, world, local, dev, None)

    # ---- C5 microbench (BASELINE.json configs[4]): GAE / VecNormalize / loss kernels over a 16 M-transition buffer
    microbench = None
    if rank == 0 and world == 1 and args.microbench:
        c.close()
        c = None
        microbench = c5_microbench(hbm_peak)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        total, threads, r, e = time_cpu_update(args.workload, 2)
        cpu_baseline = {"value": n_batch_local / total, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"full rollout ({n_steps} steps x {n_envs} envs, {r:.2f} s) + 2 of {epochs} epochs ({e:.2f} s/epoch), "
                                  f"train time scaled to {epochs} epochs", "update_samples_per_sec": n_batch_local / e}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args.workload, world),
            "update_samples_per_sec": upd_sps, "train_ms_per_step": ms_train / args.steps, "wall_ms_per_step": t_wall / args.steps * 1e3,
            "gpu_launches": int(ctr["kernel_launches"]), "clocks": clocks, "roofline": roofline, "kernel_ms": kernels,
            "cpu_baseline": cpu_baseline, "e2e": e2e,
        }
        if parity is not None:
            line["parity"] = parity
        if microbench is not None:
            line["microbench"] = microbench
        if c4 is not None:
            line["c4"] = c4
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if c is not None:
        c.close()
    if world > 1:
        dist.destroy_process_group()


def c4_sharded(core, rank, world, local, dev, _unused):
    """One C4 update = rollout of 64 steps x 65 536 envs + 10 epochs x 32 minibatches of 131 072 samples, [256,256], sharded."""
    import torch
    import torch.distributed as dist
    from ppo_cpp_b200.dist import setup_comm
    n_envs = 65536 // world
    c = core.PPOCore(device=local, hidden1=256, hidden2=256, n_envs=n_envs, n_steps=64, nminibatches=32, noptepochs=10, seed=1234,
                     rank=rank, world_size=world, env_offset=rank * n_envs, n_envs_global=65536)
    c.init_orthogonal(7)
    setup_comm(core, c, rank, world)
    c.shuffle_seed(42)
    c.synth_env_reset()
    stream = torch.cuda.ExternalStream(c.stream, device=dev)

    def sync():
        c.sync()
        torch.cuda.synchronize()
        dist.barrier()

    for _ in range(2):
        c.rollout_synthetic()
        c.train_update(LR, CLIPRANGE, want_losses=False)
    sync()
    c.counters(reset=True)
    K = 3
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for e0, e1, em in evs:
        e0.record(stream)
        c.rollout_synthetic()
        em.record(stream)
        c.train_update(LR, CLIPRANGE, want_losses=False)
        e1.record(stream)
    sync()
    ctr = c.counters()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b, _ in evs), sum(m.elapsed_time(b) for _, b, m in evs)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    fam = c.kernel_family("train")
    err = c.comm_error()
    c.close()
    nb = 65536 * 64
    ms, ms_train = float(t[0]) / K, float(t[1]) / K
    return {"workload": "C4: 65536 envs, MLP [256,256], 4194304 transitions per update, sharded over %d GPUs (strong scaling)" % world,
            "n_envs_per_gpu": n_envs, "minibatch_per_gpu": nb // 32 // world, "steps": K, "warmup": 2, "ms_per_step": ms, "train_ms_per_step": ms_train,
            "value": nb / (ms * 1e-3), "unit": UNIT, "update_samples_per_sec": nb * 10 / (ms_train * 1e-3), "kernel_family": fam,
            "train_tflops_algorithmic": nb * 10 * train_flops_per_sample(18, 18, 256, 256) / (ms_train * 1e-3) / 1e12,
            "gpu_launches": int(ctr["kernel_launches"]), "graph_launches": int(ctr["graph_launches"]), "mailbox_timeout": bool(err)}


def multi_gpu_parity(rank, world, local, hidden):
    """tests/mgpu_check.py's comparison at the bench's world size, for the bench's net: 2 updates of 48 envs per rank x 32
    steps sharded over `world` ranks vs the same 48 x world envs on one GPU; then every rank's parameters against rank 0's."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import mgpu_check
    sharded = mgpu_check.run(world, rank, local, 48, hidden, p2p=True)
    out = None
    if rank == 0:
        single = mgpu_check.run(1, 0, local, 48 * world, hidden)
        scale = float(np.abs(single["params"]).max())
        out = {"case": f"hidden {list(hidden)}, 48 envs/rank x 32 steps, 2 updates, peer-mailbox path",
               "sharded_vs_single_gpu_param_rel_diff": float(np.abs(sharded["params"] - single["params"]).max() / scale),
               "sharded_vs_single_gpu_loss_abs_diff": float(np.abs(sharded["losses"] - single["losses"]).max()),
               "vecnorm_counts_equal": bool(sharded["stats"]["obs_count"] == single["stats"]["obs_count"])}
    t = torch.tensor(sharded["params"], device=f"cuda:{local}")
    ref = t.clone()
    dist.broadcast(ref, 0)
    flags = [None] * world
    dist.all_gather_object(flags, bool(torch.equal(t, ref)))
    if rank == 0:
        out["replicas_bit_identical"] = all(flags)
    return out


def c5_microbench(hbm_peak):
    """Each kernel of the path alone over a 65 536-env x 256-step buffer (16.8 M transitions, 2.8 GB: far larger than L2),
    CUDA events on the core's stream, algorithmic bytes (SURVEY §8d) against the measured HBM copy bandwidth."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import microbench_c5
    rows = microbench_c5.measure(65536, 256, 4, 5, hbm_peak, 10)
    return {"workload": "C5: 65536 envs x 256 steps = 16.8 M transitions, MLP [4,5]", "peak_gbs": hbm_peak,
            "kernels": [{k: r[k] for k in ("kernel", "units_per_launch", "bytes_per_unit", "ms", "achieved_gbs", "frac")} for r in rows]}


def main():
    def positive(s):
        if int(s) < 1:
            raise argparse.ArgumentTypeError("must be at least 1")
        return int(s)

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive, default=50, help="timed PPO updates")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-e2e", dest="e2e", action="store_false")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-microbench", dest="microbench", action="store_false")
    ap.add_argument("--no-parity", dest="parity", action="store_false")
    ap.add_argument("--no-c4", dest="c4", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
