"""Cost of shared statistics (VectorTrainer(stats_group=...), EnvBatch.share_stats): collect() with per-rank statistics
against collect() with statistics shared over a process group, and the cross-rank fold (sat_stats_fold) alone.

    python tools/time_shared_stats.py [--reps 5]                    # one process: a 1-rank NCCL group
    torchrun --nproc-per-node G tools/time_shared_stats.py          # G GPUs: the shared mode pays the all_gather

collect(): two trainers of the same size, seeds and weights (cw mode, starts mode, reward scaling and observation
normalisation on), one per-rank and one shared; their collect() calls alternate, a device synchronise before and after
each, and the report is the median over --reps calls of the wall time per step. At 8192 envs x T = 256 and 65 536 envs x
T = 64. The shared step is sat_env_step_partials + all_gather_into_tensor + sat_stats_fold in place of sat_env_step.
Under torchrun, each rank holds the given number of envs (the union is G times larger) and also reports the
all_gather of one step's partials alone (CUDA events, 200 calls).
fold: sat_stats_fold over G = 1, 2, 4, 8 gathered shards of 65 536 envs (random partials, G * 1024 blocks x 19 dims),
CUDA events around 500 calls after 50 warm-up calls; the partials (at most 2.5 MB) stay in L2.
Prints the card name and power limit and one JSON line per measurement (rank 0). Writes nothing."""
import argparse
import json
import os
import subprocess
import sys
import time
import types

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppo_rl_satellite_b200 import engine as eng  # noqa: E402
from ppo_rl_satellite_b200 import rollout  # noqa: E402
from ppo_rl_satellite_b200.dropin import ppo_continuous as P  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def box():
    c = np.array([200000.0, 0, 0, 0, 0, 0, 18000.0, 0, 0, 0, 0, 0])
    d = np.array([50000.0] * 3 + [3.0] * 3 + [50000.0] * 3 + [3.0] * 3)
    return c - d, c + d


def args(B):
    return types.SimpleNamespace(policy_dist="Gaussian", max_action=1.6, batch_size=B, mini_batch_size=4096,
                                 max_train_steps=int(3e6), lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1,
                                 K_epochs=1, entropy_coef=0.01, set_adam_eps=True, use_grad_clip=True, use_lr_decay=True,
                                 use_adv_norm=True, state_dim=18, action_dim=3, hidden_width=256, use_tanh=1,
                                 use_orthogonal_init=True, chkpt_dir="/tmp")


def trainer(n, T, rank, group):
    env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=200, start_box=box(), start_seed=3,
                       row_offset=rank * n)
    torch.manual_seed(0)
    agent, opp = P.PPO_continuous(args(n * T), "pursuer"), P.PPO_continuous(args(n * T), "evader")
    return rollout.VectorTrainer(env, agent, opp, T, rank=rank, seed=1, stats_group=group)


def time_collect(n, T, reps, rank, group):
    trs = {"per_rank": trainer(n, T, rank, None), "shared": trainer(n, T, rank, group)}
    times = {k: [] for k in trs}
    for i in range(reps + 1):
        for k in (("per_rank", "shared") if i % 2 == 0 else ("shared", "per_rank")):
            dist.barrier(group)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            trs[k].collect()
            torch.cuda.synchronize()
            if i:                                         # the first round warms up both
                times[k].append((time.perf_counter() - t0) / T * 1e6)
    same = torch.equal(trs["per_rank"].buf.rew64, trs["shared"].buf.rew64)
    return {k: float(np.median(v)) for k, v in times.items()}, {k: float(np.min(v)) for k, v in times.items()}, same


def time_events(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def time_fold(G, n=65536):
    blocks = (n + 63) // 64
    g = torch.Generator(device="cuda").manual_seed(G)
    gathered = torch.rand((G, blocks * 19 * 2), generator=g, dtype=torch.float64, device="cuda") + 1.0
    rank_rows = torch.full((G,), n, dtype=torch.int64, device="cuda")
    ws = torch.zeros(256, dtype=torch.uint8, device="cuda")
    obs, ret = eng.RunningStats(18), eng.RunningStats(1)
    std = torch.zeros(1, dtype=torch.float64, device="cuda")
    return time_events(lambda: eng.fold_stats(gathered, rank_rows, 0, obs, ret, std, ws), 500, 50)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if "WORLD_SIZE" in os.environ:
        local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
        dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % (29500 + os.getpid() % 1000), rank=0,
                                world_size=1, device_id=torch.device("cuda", 0))
    rank, world = dist.get_rank(), dist.get_world_size()
    group = dist.group.WORLD
    out = []
    try:
        name, lim = card()
        if rank == 0:
            print(f"# {name}, power limit / max SM clock: {lim}; {world} rank(s), NCCL", flush=True)
        for n, T in ((8192, 256), (65536, 64)):
            med, best, same = time_collect(n, T, a.reps, rank, group)
            rec = {"what": "collect_us_per_step", "envs_per_rank": n, "T": T, "ranks": world, "median": med, "min": best,
                   "rewards_equal": same}
            if world > 1:
                ex = eng.StatsExchange(group, n, 0, torch.device("cuda", torch.cuda.current_device()))
                rec["all_gather_us"] = time_events(
                    lambda: dist.all_gather_into_tensor(ex.gathered.view(-1), ex.send, group=group), 200, 20)
            out.append(rec)
        if rank == 0:
            for G in (1, 2, 4, 8):
                out.append({"what": "fold_us", "G": G, "envs_per_shard": 65536, "us": time_fold(G)})
            for rec in out:
                rec.update(gpu=name, power_limit_max_sm_clock=lim)
                print(json.dumps(rec), flush=True)
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
