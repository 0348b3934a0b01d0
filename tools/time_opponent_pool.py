"""Opponent-pool launch (sat_actor_sample_pool_tc: learner + K snapshots in one persistent grid) against the pair launch
(sat_actor_sample_pair_tc) and against K per-group launches, on fp32 observations and on the env-state path, at 8192 and
65 536 rows; then VectorTrainer.collect() us/step with and without a pool. Prints the card's name and power limit of the run.

    python tools/time_opponent_pool.py [--reps 40] [--out result.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppo_rl_satellite_b200 import engine as eng, rollout  # noqa: E402
import bench  # noqa: E402

L = eng.L


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


FLUSH = None


def timed(fn, reps):
    """mean device time (us) of fn over reps launches after 5 warm-ups; L2 overwritten before every timed launch"""
    ts = []
    for i in range(reps + 5):
        FLUSH.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(i); e1.record(); e1.synchronize()
        if i >= 5:
            ts.append(e0.elapsed_time(e1))
    return float(np.mean(ts)) * 1e3


def launches(reps):
    lib = L.load()
    learner = eng.GaussianActorKernel().load_state_dict(bench.orthogonal_actor_state(torch, 0))
    other = eng.GaussianActorKernel().load_state_dict(bench.orthogonal_actor_state(torch, 1))
    pool = eng.OpponentPool(16)
    for k in range(16):
        pool.add(eng.GaussianActorKernel().load_state_dict(bench.orthogonal_actor_state(torch, 10 + k)))
    rows = []
    for n in (8192, 65536):
        obs = torch.randn((n, 18), device="cuda")
        env = eng.EnvBatch(n, mode="cw")
        st = eng.RunningStats(18)
        st.update_normalize(env.observe())
        out = [torch.empty((n, 3), device="cuda") for _ in range(4)]
        img_b = torch.empty(L.ACTOR_TC_IMAGE_FLOATS, device="cuda")
        for path in ("fp32", "state"):
            o = (L.ptr(obs), None, None) if path == "fp32" else (None, C.byref(env.st), L.ptr(st.buf))

            def pair(i):
                L.check(lib.sat_actor_sample_pair_tc(C.byref(learner.w), C.byref(other.w), learner._image().data_ptr(),
                                                     img_b.data_ptr(), *o, n, 0, 1, i, i, L.ptr(out[0]), L.ptr(out[1]), None,
                                                     L.ptr(out[2]), L.ptr(out[3]), L.stream_ptr()), "pair")
            t_pair = timed(pair, reps)
            for K in (1, 4, 8, 16):
                ends = rollout.pool_group_bounds(n, K)
                arr = (L.SatActorPoolGroup * K)()
                for k, e in enumerate(ends):
                    arr[k] = pool.group(k)
                    arr[k].row_end = e

                def one(i):
                    L.check(lib.sat_actor_sample_pool_tc(C.byref(learner.w), learner._image().data_ptr(), arr, K, *o, n, 0, 1,
                                                         i, i, L.ptr(out[0]), L.ptr(out[1]), None, L.ptr(out[2]),
                                                         L.ptr(out[3]), L.stream_ptr()), "pool")
                subs = []
                lo = 0
                for e in ends:
                    sub = L.SatEnvState(env._state_buf.data_ptr() + 8 * lo, env._istate_buf.data_ptr() + 4 * lo, e - lo, env.ld)
                    subs.append((lo, e, sub))
                    lo = e

                def per_group(i):
                    L.check(lib.sat_actor_sample_tc(C.byref(learner.w), learner._image().data_ptr(), *o, n, 0, 1, i, None,
                                                    L.ptr(out[0]), L.ptr(out[1]), None, None, None, L.stream_ptr()), "learner")
                    for k, (lo, e, sub) in enumerate(subs):
                        kk = pool.kernel(k)
                        src = (L.ptr(obs[lo:e]), None, None) if path == "fp32" else (None, C.byref(sub), L.ptr(st.buf))
                        L.check(lib.sat_actor_sample_tc(C.byref(kk.w), kk._image().data_ptr(), *src, e - lo, lo, 1, i, None,
                                                        L.ptr(out[2][lo:e]), L.ptr(out[3][lo:e]), None, None, None,
                                                        L.stream_ptr()), "group")
                t_pool, t_groups = timed(one, reps), timed(per_group, reps)
                r = dict(rows=n, path=path, K=K, pair_us=t_pair, pool_us=t_pool, per_group_us=t_groups,
                         pool_over_pair=t_pool / t_pair)
                rows.append(r)
                print(f"rows {n:6d} {path:5s} K {K:2d}: pair {t_pair:7.1f} us  pool {t_pool:7.1f} us ({t_pool / t_pair:5.3f} x pair)"
                      f"  learner + {K} per-group launches {t_groups:7.1f} us", flush=True)
    return rows


def _args(B, mb):
    return types.SimpleNamespace(policy_dist="Gaussian", max_action=1.6, batch_size=B, mini_batch_size=mb, max_train_steps=int(3e6),
                                 lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1, K_epochs=1, entropy_coef=0.01,
                                 set_adam_eps=True, use_grad_clip=True, use_lr_decay=False, use_adv_norm=True, state_dim=18,
                                 action_dim=3, hidden_width=256, use_tanh=1, use_orthogonal_init=True, chkpt_dir="/tmp")


def collects(K=8):
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    rows = []
    for n, T in ((8192, 256), (65536, 64)):
        res = {}
        for use_pool in (False, True):
            torch.manual_seed(0)
            agent, opp = P.PPO_continuous(_args(n * T, 4096), "pursuer"), P.PPO_continuous(_args(n * T, 4096), "evader")
            pool = None
            if use_pool:
                opp.sync_kernels()
                pool = eng.OpponentPool(K)
                for _ in range(K):
                    pool.add(opp.actor_kernel)
            tr = rollout.VectorTrainer(eng.EnvBatch(n, mode="cw"), agent, opp, T, seed=1, opponent_pool=pool)
            tr.collect()                                   # warm-up
            ts = []
            for _ in range(3):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); tr.collect(); e1.record(); e1.synchronize()
                ts.append(e0.elapsed_time(e1) * 1e3 / T)
            res[use_pool] = float(np.median(ts))
            del tr
        rows.append(dict(envs=n, T=T, K=K, no_pool_us_per_step=res[False], pool_us_per_step=res[True]))
        print(f"collect() {n} envs x {T} steps: {res[False]:7.1f} us/step without a pool, {res[True]:7.1f} us/step with "
              f"a pool of {K}", flush=True)
    return rows


def main():
    global FLUSH
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # larger than the 126 MB L2
    c = card()
    print(f"card: {c}", flush=True)
    res = {"card": c, "launches": launches(a.reps), "collect": collects()}
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
