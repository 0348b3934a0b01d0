#!/usr/bin/env python
"""bench.py -- throughput of the batched satellite environment step on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric (BASELINE.json): RK4 satellite env-steps/sec on synthetic random orbits and actions. A "step" is
one pass of the hot path over one batch: one fused env step in rk4 mode (clip/gate/impulse, S RK4+J2
substeps of both craft, terminal checks, danger-zone count, reward, observation/return running statistics,
auto-reset) for every env of the batch, with the step's actions already resident in HBM (`value`) or
arriving in host buffers through the reference-facing step(pa, ea) call (`e2e`). The same step with the
two fused Gaussian actors sampling the actions on the device (config 3 "with fused actor sampling") is
reported beside it as `config3_full_step` (with its own roofline, the fp32 actor kernel).

N = 1 workload: BASELINE config 3 (65 536 envs, S = 100 substeps of h = 1 s, J2 on). N > 1: the same
per-GPU batch on every rank (weak scaling; envs are independent, no data-path collective); in addition `config4`
(1 048 576 envs / N per GPU, horizon-256 on-device rollout) and, at N = 8, the PPO section at config 5's
2048-step horizon.

One JSON line on stdout (rank 0). See DESIGN.md "Measurement" for every field.

--dump-outputs DIR writes what rank 0's last timed step returned to its caller: obs.npy (next observations, fp32,
[envs, 18]), reward.npy (fp64), done.npy (0 / 1 as fp32) and ret_std.npy (std of the discounted returns, fp64). The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_ENV_STEP = 34800.0        # SURVEY.md s8d: 2 craft x 100 substeps x 174 FLOP (RK4 + J2), fp64
FLOP_RK4_J2 = 174.0
FP64_INSTR_RK4_J2 = 106.5      # DFMA+DMUL+DADD per RK4+J2 step in the SASS of rk4_kernel<true,2> (cuobjdump, DESIGN.md s4)
FLOP_ACTOR = 141824.0          # fp32 per actor forward
# one sample through one PPO optimiser step (both networks): forward 141 824 + 140 800, backward through fc2 2 x 131 072,
# weight gradients 2 x 2 x (256 x 256 + 18 x 256) + heads  (DESIGN.md s5b)
FLOP_PPO_SAMPLE_STEP = (141824.0 + 140800.0) + 2 * 131072.0 + 2 * 2 * (65536.0 + 4608.0) + 2 * 4 * 256.0
BYTES_ENV_STEP = 345.0
BYTES_GAE_SAMPLE = 17.0        # SURVEY.md s8d: r 4 + v 4 + done 1 + adv 4 + v_target 4
SM_COUNT, SM_GHZ = 148, 1.965
FP64_NOMINAL_TFLOPS = SM_COUNT * 64 * 2 * SM_GHZ / 1e3      # 37.2: 64 DFMA lanes per SM
FP32_NOMINAL_TFLOPS = SM_COUNT * 128 * 2 * SM_GHZ / 1e3     # 74.5: 128 FFMA lanes per SM


def ncu_traffic(kernel, n_envs):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/ncu_traffic.json: dram__bytes_read.sum +
    dram__bytes_write.sum of one `ncu --set full` launch), scaled to this run's env count; the file names the capture."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        rec = json.load(open(path))[kernel]
    except Exception:
        return None, "profiles/ncu_traffic.json has no entry for " + kernel
    return rec["dram_bytes_per_launch"] * (n_envs / rec["envs"]), f"{rec['source']} ({rec['captured']}), {rec['envs']} envs, scaled by n"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3, help="untimed warm-up steps (at least 3 are always run)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--substeps", type=int, default=100)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ppo", action="store_true", help="skip the PPO samples/sec section")
    ap.add_argument("--ppo-horizon", type=int, default=256, help="rollout horizon T of the PPO section (config 5: 2048)")
    ap.add_argument("--ppo-envs", type=int, default=8192, help="envs per GPU of the PPO section (config 5: 65536/8)")
    ap.add_argument("--ppo-minibatch", type=int, default=65536, help="samples per GPU per optimiser step")
    ap.add_argument("--ppo-eager", action="store_true", help="run the optimiser steps eagerly instead of as a CUDA graph")
    ap.add_argument("--ppo-update", choices=("fused", "torch"), default="fused",
                    help="optimiser step: hand-written forward/backward/Adam kernels, or the PyTorch step (CUDA-graphed)")
    ap.add_argument("--cpu-sample-envs", type=int, default=0, help="0 = auto (about 10-20 s of CPU work)")
    ap.add_argument("--config4", action="store_true", help="also run BASELINE config 4 at N=1 (1 048 576 envs on one GPU); "
                                                           "always run for N>1 (1 048 576 / N envs per GPU, T=256)")
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0) as DIR/<name>.npy; "
                                                           "bench_outputs/ in the tree is git-ignored")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup_requested = args.warmup
    if args.gpus >= 8 and "--ppo-horizon" not in " ".join(sys.argv):
        args.ppo_horizon = 2048                  # config 5 proper: 2048-step x 65 536-env rollout on 8 GPUs (8192 envs/GPU)
    args.warmup = max(3, args.warmup)            # timing rule: never fewer than 3 untimed warm-up steps
    return args


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_env_steps_per_s(n_envs, steps, substeps, nthreads):
    """Times the CPU restatement of the same workload (oracle port of the reference's env logic + the RK4
    script's integrator) on the host cores: returns env-steps/s."""
    from oracle import oracle as O
    env = O.BatchEnv(n_envs, d_capture=20000.0, max_episode_steps=1000, nthreads=nthreads)
    rng = np.random.default_rng(1)
    pa = rng.uniform(-2, 2, (n_envs, 3)).astype(np.float32).astype(np.float64)
    ea = rng.uniform(-2, 2, (n_envs, 3)).astype(np.float32).astype(np.float64)
    env.step_rk4(pa, ea, substeps=substeps)                      # warm-up
    t0 = time.perf_counter()
    for _ in range(steps):
        env.step_rk4(pa, ea, substeps=substeps)
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, dt


def reference_python_rows():
    """BASELINE.md s3 rows timed with the reference's OWN Python code (unmodified files staged in the git-ignored baseline/_ref
    by tools/stage_reference.py) on this box's host cores: C-env-1, C-rk4-scalar, C-rk4-batch, C-actor, C-gae, C-update.
    Bounded to ~2 s per row. Returns None when the staged reference is absent."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref, "environment.py")):
        return None
    import contextlib, io
    os.environ["SAT_REFERENCE_DIR"] = ref
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        import refshim
        import torch
        mods = refshim.load()
        rows = {"source": "unmodified reference files in baseline/_ref (tools/stage_reference.py), python %s, numpy %s, torch %s, "
                          "torch threads %d" % (sys.version.split()[0], np.__version__, torch.__version__, torch.get_num_threads())}
        rng = np.random.default_rng(1)

        def timed(fn, budget=2.0, min_iters=3):
            n_, t0 = 0, time.perf_counter()
            while True:
                fn(); n_ += 1
                dt = time.perf_counter() - t0
                if n_ >= min_iters and dt >= budget:
                    return n_ / dt, n_, dt
        # C-env-1: env.step (Flag 0, CW propagation + danger zone + reward) as shipped, stdout suppressed, 1 core
        env = refshim.make_env(20000, 1000)
        env.reset(0)
        cnt = [0]
        def env_step():
            cnt[0] += 1
            _, _, d = refshim.quiet_step(env, rng.uniform(-2, 2, 3), rng.uniform(-2, 2, 3), cnt[0])
            if d:
                env.reset(0); cnt[0] = 0
        for _ in range(50):
            env_step()
        rate, k, dt = timed(env_step)
        rows["C-env-1"] = {"value": rate, "unit": "env-steps/s", "cores": 1, "sample": f"{k} reference env.step calls (cw mode as shipped), {dt:.1f} s",
                           "code": "environment.py:81-179"}
        # C-rk4-scalar / C-rk4-batch: the script's RungeKutta (lines 9-40 executed unmodified)
        ns = refshim.load_rk4_script()
        x1 = np.array([6678.137, 0.0, 0.0, 0.0, 6.789530297, 3.686414173])
        st = {"x": x1}
        def rk_scalar():
            st["x"] = ns["RungeKutta"](0.0, st["x"], 1.0)
        rate, k, dt = timed(rk_scalar, budget=1.5)
        rows["C-rk4-scalar"] = {"value": rate, "unit": "RK4 steps/s", "cores": 1, "sample": f"{k} scalar RungeKutta calls, {dt:.1f} s",
                                "code": "RK4 script :15-40"}
        ang = rng.uniform(0, 2 * np.pi, 4096)
        xb = np.array([7000 * np.cos(ang), 7000 * np.sin(ang), rng.uniform(-500, 500, 4096), -7.5 * np.sin(ang), 7.5 * np.cos(ang), rng.uniform(-.5, .5, 4096)])
        stb = {"x": xb}
        def rk_batch():
            stb["x"] = ns["RungeKutta"](0.0, stb["x"], 1.0)
        rate, k, dt = timed(rk_batch, budget=1.5)
        rows["C-rk4-batch"] = {"value": rate * 4096, "unit": "RK4 steps/s", "cores": 1, "sample": f"{k} RungeKutta calls on a (6, 4096) array, {dt:.1f} s",
                               "code": "RK4 script :15-40"}
        # C-actor / C-gae / C-update: the reference's PPO_continuous
        P = mods["ppo_continuous"]
        a = _PpoArgs(policy_dist="Gaussian", max_action=1.6, batch_size=2048, mini_batch_size=64, max_train_steps=int(3e6),
                     lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1, K_epochs=10, entropy_coef=0.01, set_adam_eps=True,
                     use_grad_clip=True, use_lr_decay=True, use_adv_norm=True, state_dim=18, action_dim=3, hidden_width=256,
                     use_tanh=True, use_orthogonal_init=True, chkpt_dir="/tmp", max_episode_steps=1000)
        with contextlib.redirect_stdout(io.StringIO()):
            agent = P.PPO_continuous(a, "pursuer")
        s1 = rng.normal(0, 1, 18)
        rate, k, dt = timed(lambda: agent.choose_action(s1), budget=1.5)
        rows["C-actor"] = {"value": rate, "unit": "choose_action calls/s (batch 1)", "cores": torch.get_num_threads(),
                           "sample": f"{k} calls, {dt:.1f} s", "code": "ppo_continuous.py:176-189"}
        xb_ = torch.randn(65536, 18)
        with torch.no_grad():
            rate, k, dt = timed(lambda: agent.actor(xb_), budget=1.5)
        rows["C-actor-batch"] = {"value": rate * 65536, "unit": "actor forwards/s on a [65536, 18] tensor", "cores": torch.get_num_threads(),
                                 "sample": f"{k} forwards, {dt:.1f} s", "code": "ppo_continuous.py:83-95"}
        RB = mods["replaybuffer"].ReplayBuffer
        rb = RB(a)
        for i in range(2048):
            rb.store(rng.normal(0, 1, 18), rng.uniform(-1, 1, 3), rng.normal(-1, .1, 3), rng.normal(), rng.normal(0, 1, 18), (i % 1000) == 999, (i % 1000) == 999)
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            agent.update(rb, 0)
        dt = time.perf_counter() - t0
        rows["C-update"] = {"value": 2048 / dt, "unit": "rollout samples/s through one update (2048 / 64 / K=10, GAE block included)",
                            "cores": torch.get_num_threads(), "sample": f"1 update, {dt:.2f} s", "code": "ppo_continuous.py:191-242"}
        # C-gae: the reference's GAE block alone (:198-210), exec'd on the same buffer
        s_, a_, lp_, r_, sn_, dw_, dn_ = rb.numpy_to_tensor()
        def gae_block():
            adv, gae = [], 0
            with torch.no_grad():
                vs, vsn = agent.critic(s_), agent.critic(sn_)
                deltas = r_ + a.gamma * (1.0 - dw_) * vsn - vs
                for delta, d in zip(reversed(deltas.flatten().numpy()), reversed(dn_.flatten().numpy())):
                    gae = delta + a.gamma * a.lamda * gae * (1.0 - d)
                    adv.insert(0, gae)
                adv = torch.tensor(adv, dtype=torch.float).view(-1, 1)
                return adv + vs
        rate, k, dt = timed(gae_block, budget=1.0)
        rows["C-gae"] = {"value": rate * 2048, "unit": "samples/s", "cores": 1, "sample": f"{k} passes of the GAE block over 2048 samples, {dt:.1f} s",
                         "code": "ppo_continuous.py:198-210"}
        return rows
    except Exception as e:                                   # a reported baseline must never break the GPU line
        return {"error": repr(e)}
    finally:
        sys.path.remove(os.path.join(ROOT, "tests"))


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_envs = args.cpu_sample_envs or 64 * cores
    # size the sample: one probe step, then as many envs as fit ~3 s per timed step
    rate, _ = cpu_env_steps_per_s(min(n_envs, 8 * cores), 1, args.substeps, cores)
    n_envs = int(max(cores, min(args.envs, rate * 3.0)))
    times = []
    from oracle import oracle as O
    env = O.BatchEnv(n_envs, d_capture=20000.0, max_episode_steps=1000, nthreads=cores)
    rng = np.random.default_rng(1)
    for i in range(args.warmup + args.steps):
        pa = rng.uniform(-2, 2, (n_envs, 3)).astype(np.float32).astype(np.float64)
        ea = rng.uniform(-2, 2, (n_envs, 3)).astype(np.float32).astype(np.float64)
        t0 = time.perf_counter()
        env.step_rk4(pa, ea, substeps=args.substeps)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.mean(times))
    value = n_envs / (ms * 1e-3)
    line = {"impl": "reference", "metric": "rk4_env_steps_per_sec", "value": value, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args, None),
            "note": "the reference is pure Python and cannot travel to the GPU box; this arm times the CPU oracle port (C, OpenMP, "
                    "literal restatement incl. MINPACK hybrd) of the same env step on all host threads",
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                             "sample": f"{n_envs} envs x {args.steps} steps (S={args.substeps} RK4+J2 substeps, env step only, actions given)"},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def config_dict(args, value):
    """the `config` object of the JSON line: identical keys (and values) in both arms so the driver can compare them"""
    return {"workload": workload_name(args), "envs_per_gpu": args.envs, "substeps": args.substeps, "h": 1.0, "j2": True,
            "l2": "flushed between timed steps (256 MiB memset outside the event pairs)",
            "timing": "CUDA events per step on the launch stream, sum over steps, max over ranks (reference arm: wall clock per step)"}


def workload_name(args):
    return (f"config3: {args.envs} envs/GPU, fused env step in rk4 mode on synthetic random orbits and actions "
            f"(S={args.substeps} x h=1s RK4 two-body+J2 of both craft, clip/gate/impulse, terminal checks, danger-zone count, "
            f"reward, running obs/return statistics, auto-reset)")


# ------------------------------------------------------------------------------------------------ ours
def orthogonal_actor_state(torch, seed):
    """random-init weights of the reference's Actor_Gaussian (orthogonal init, ppo_continuous.py:76-81)."""
    g = torch.Generator().manual_seed(seed)
    def orth(rows, cols, gain):
        w = torch.empty(rows, cols)
        torch.nn.init.orthogonal_(w, gain=gain, generator=g)
        return w
    return {"fc1.weight": orth(256, 18, 1.0), "fc1.bias": torch.zeros(256), "fc2.weight": orth(256, 256, 1.0),
            "fc2.bias": torch.zeros(256), "mean_layer.weight": orth(3, 256, 0.01), "mean_layer.bias": torch.zeros(3),
            "log_std": torch.zeros(1, 3)}


class _PpoArgs:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def run_ppo_section(args, rank, world, dev, torch, dist, eng):
    """config 5 per-GPU share: T x n on-device rollout (2 actors + env step in rk4 mode), critic values, GAE kernel,
    advantage normalisation with all-reduced moments, K = 10 epochs of minibatch PPO with NCCL gradient all-reduce."""
    from ppo_rl_satellite_b200 import rollout
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    T, n, mb = args.ppo_horizon, args.ppo_envs, args.ppo_minibatch
    a = _PpoArgs(policy_dist="Gaussian", max_action=1.6, batch_size=T * n, mini_batch_size=mb, max_train_steps=int(3e6),
                 lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1, K_epochs=10, entropy_coef=0.01,
                 set_adam_eps=True, use_grad_clip=True, use_lr_decay=True, use_adv_norm=True, state_dim=18, action_dim=3,
                 hidden_width=256, use_tanh=True, use_orthogonal_init=True, chkpt_dir="/tmp")   # CPPO_main.py:14-39 defaults
    torch.manual_seed(0)                                              # identical initial weights on every rank
    env = eng.EnvBatch(n, mode="rk4", substeps=args.substeps, h=1.0, d_capture=20000.0, max_episode_steps=1000, device=dev)
    agent, opp = P.PPO_continuous(a, "pursuer", device=dev), P.PPO_continuous(a, "evader", device=dev)
    tr = rollout.VectorTrainer(env, agent, opp, T, rank=rank)
    group = None if world > 1 else False

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    use_graph = not args.ppo_eager and (world == 1 or os.environ.get("SAT_GRAPH_DDP", "1") == "1")
    fused = args.ppo_update == "fused"
    tr.collect(); tr.update(mb, group=group, use_graph=use_graph, fused=fused)     # warm-up iteration (workspaces, graph capture)
    sync()
    t0 = time.perf_counter(); tr.collect(); sync(); t1 = time.perf_counter()
    tr.update(mb, total_steps=1, group=group, use_graph=use_graph, fused=fused); sync(); t2 = time.perf_counter()
    dt = torch.tensor([t1 - t0, t2 - t1], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    tc, tu = float(dt[0]), float(dt[1])
    samples = T * n * world
    return {"ppo_samples_per_sec": samples / (tc + tu), "rollout_s": tc, "update_s": tu, "samples": samples,
            "config": f"T={T} x {n} envs/GPU (rk4 mode, S={args.substeps}), minibatch {mb}/GPU, K=10, gamma .99, lambda .95 "
                      f"(CPPO_main.py:24-27); config 5 proper is --ppo-horizon 2048 --ppo-envs 8192 on 8 GPUs",
            "optimizer_steps": 10 * -(-T * n // mb), "update_impl": ("fused CUDA kernels, actor and critic chains on two streams: forward/backward (csrc/ppo_fb_tc.cu) and dW2 "
                                                                 "(csrc/ppo_wgrad2_tc.cu) on the tensor cores as exact bf16x3 splits, dW1 / partial sums / Adam fp32 (csrc/ppo_update.cu)"
                                                                 if eng.L.load().sat_ppo_use_tensor_cores(-1) else
                                                                 "fused CUDA kernels, fp32 FFMA2 (csrc/ppo_update.cu; SAT_PPO_TC=0), actor and critic chains on two streams")
                                                                if fused else "PyTorch autograd + torch.optim.Adam",
            "cuda_graph": bool(not fused and use_graph and agent._graph is not None), "allreduce": None if world == 1 else (
                "fused into the Adam kernel: every rank reads all ranks' flat gradients (286 KB + 284 KB) from NVLink peer memory "
                "(torch symmetric memory) in rank order after a device-side barrier; no NCCL call on the step"
                if fused and agent._fused is not None and any(agent._fused.get("peers", {}).values()) else "NCCL, 2 flat buckets (286 KB + 284 KB) per step"),
            "timing": "wall clock with barrier + synchronize on both sides, max over ranks"}


def run_config4(args, rank, world, dev, torch, dist, eng):
    """BASELINE config 4: 1 048 576 envs split evenly over the ranks (524 288 / 262 144 / 131 072 per GPU), rk4 mode with J2,
    S substeps, rollout horizon T = 256 with both actors sampling on the device and every transition stored (time-major
    rollout buffer, 153 B/sample). Philox counters use the global env id, no collective. Device time, max over ranks."""
    from ppo_rl_satellite_b200 import rollout
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    total, T = 1 << 20, 256
    lo, hi = rollout.shard_bounds(total, world, rank)
    n = hi - lo
    a = _PpoArgs(policy_dist="Gaussian", max_action=1.6, batch_size=T * n, mini_batch_size=65536, max_train_steps=int(3e6),
                 lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1, K_epochs=10, entropy_coef=0.01,
                 set_adam_eps=True, use_grad_clip=True, use_lr_decay=True, use_adv_norm=True, state_dim=18, action_dim=3,
                 hidden_width=256, use_tanh=True, use_orthogonal_init=True, chkpt_dir="/tmp")
    torch.manual_seed(0)
    env = eng.EnvBatch(n, mode="rk4", substeps=args.substeps, h=1.0, d_capture=20000.0, max_episode_steps=1000, device=dev)
    rng = np.random.default_rng(4321 + rank)
    env.set_state(np.array([200000.0, 0, 0]) + rng.normal(0, 3e4, (n, 3)), rng.normal(0, 3.0, (n, 3)),
                  np.array([18000.0, 0, 0]) + rng.normal(0, 3e4, (n, 3)), rng.normal(0, 3.0, (n, 3)))
    agent, opp = P.PPO_continuous(a, "pursuer", device=dev), P.PPO_continuous(a, "evader", device=dev)
    tr = rollout.VectorTrainer(env, agent, opp, T, rank=0)
    tr.row_offset = lo                                           # Philox counter = global env id (shard-invariant)
    warm = rollout.VectorTrainer(env, agent, opp, 4, rank=0)
    warm.row_offset = lo
    warm.collect()
    del warm
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); tr.collect(); e1.record(); e1.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    # the same rollout with the fp32 FFMA2 actor kernels (csrc/actor.cu; SAT_ACTOR_TC=0), see config3_full_step
    tc_was = agent.actor_kernel.use_tc
    agent.actor_kernel.use_tc = opp.actor_kernel.use_tc = False
    e0.record(); tr.collect(); e1.record(); e1.synchronize()
    ms_ff = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_ff, op=dist.ReduceOp.MAX)
    ms_ff = float(ms_ff.item())
    agent.actor_kernel.use_tc = opp.actor_kernel.use_tc = tc_was
    out = {"what": "1 048 576 envs / %d GPUs = %d envs per GPU, rk4 mode (S=%d, J2 on), T=256 on-device rollout: 2 actor samplings + env "
                   "step per time step, transitions stored time-major; no collective; CUDA events around the rollout, max over ranks" % (world, n, args.substeps),
           "envs_total": total, "envs_per_gpu": n, "horizon": T, "rollout_ms": ms, "ms_per_step": ms / T,
           "env_steps_per_sec": total * T / (ms * 1e-3), "rk4_steps_per_sec": total * T / (ms * 1e-3) * 2 * args.substeps,
           "episodes_finished": int(tr.buf.done.sum().item()), "err_envs": int(env.err.sum().item()),
           "rollout_buffer_gb_per_gpu": tr.buf.bytes_per_sample * T * n / 1e9,
           "actors": "tensor cores (bf16x3, both networks in one persistent launch)" if tc_was else "fp32 FFMA2",
           "ffma2_actor_variant": {"rollout_ms": ms_ff, "ms_per_step": ms_ff / T, "env_steps_per_sec": total * T / (ms_ff * 1e-3),
                                   "what": "same rollout with the fp32 CUDA-core actor kernels (SAT_ACTOR_TC=0)"}}
    del tr, env, agent, opp
    torch.cuda.empty_cache()
    return out


DUMP_MAX_BYTES = 64_000_000


def _float_array(t):
    a = t.cpu().numpy()
    return a if a.dtype in (np.float32, np.float64) else a.astype(np.float32)


def dump_outputs(path, per_env, extra):
    """Writes a step's outputs as path/<name>.npy, float64 arrays as they are and everything else as float32, so that two
    builds can be compared output for output. When the per-env arrays exceed DUMP_MAX_BYTES, every one of them is cut to
    the same seeded sample of rows and the sampled row indices are written as rows.npy."""
    os.makedirs(path, exist_ok=True)
    per_env = {k: _float_array(v) for k, v in per_env.items()}
    extra = {k: _float_array(v) for k, v in extra.items()}
    n = len(next(iter(per_env.values())))
    row_bytes = sum(a.nbytes // n for a in per_env.values())
    if row_bytes * n > DUMP_MAX_BYTES:
        keep = (DUMP_MAX_BYTES - 1_000_000) // (row_bytes + 8)      # 8 B per row for rows.npy, 1 MB for the rest
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        per_env = {k: a[rows] for k, a in per_env.items()}
        extra["rows"] = rows.astype(np.float64)
    for k, a in {**per_env, **extra}.items():
        np.save(os.path.join(path, k + ".npy"), a)


def bind_to_gpu_numa_node(local_rank):
    """Multi-GPU runs: pin this rank (and therefore its first-touch pinned host buffers) to the CPUs NVML reports as local
    to its GPU, so the e2e path's PCIe traffic does not cross the socket interconnect. Returns the CPU count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w in range(words) for b in range(64) if (int(mask[w]) >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus and len(cpus) < os.cpu_count():
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from ppo_rl_satellite_b200 import engine as eng
    from ppo_rl_satellite_b200 import _lib as L

    numa_cpus = bind_to_gpu_numa_node(local_rank) if world > 1 and os.environ.get("SAT_NUMA_BIND", "1") != "0" else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    n = args.envs
    S = args.substeps

    env = eng.EnvBatch(n, mode="rk4", substeps=S, h=1.0, d_capture=20000.0, max_episode_steps=1000, auto_reset=True, device=dev)
    # synthetic random relative orbits around the reset geometry (different per rank / env)
    rng = np.random.default_rng(1234 + rank)
    P = np.array([200000.0, 0, 0]) + rng.normal(0, 3e4, (n, 3)); E = np.array([18000.0, 0, 0]) + rng.normal(0, 3e4, (n, 3))
    env.set_state(P, rng.normal(0, 3.0, (n, 3)), E, rng.normal(0, 3.0, (n, 3)))
    pursuer = eng.GaussianActorKernel(device=dev).load_state_dict(orthogonal_actor_state(torch, 0))
    evader = eng.GaussianActorKernel(device=dev).load_state_dict(orthogonal_actor_state(torch, 1))
    obs_stats, ret_stats = eng.RunningStats(18, dev), eng.RunningStats(1, dev)
    x0 = env.observe()
    obs_stats.update_normalize(x0)                                  # statistics of the initial observations

    RING = 8                                                        # rollout ring: obs/act/logp/reward/done per step
    buf_obs = torch.empty((RING, n, 18), dtype=torch.float32, device=dev)
    buf_act = torch.empty((RING, n, 3), dtype=torch.float32, device=dev)
    buf_logp = torch.empty((RING, n, 3), dtype=torch.float32, device=dev)
    buf_eact = torch.empty((RING, n, 3), dtype=torch.float32, device=dev)
    buf_elogp = torch.empty((RING, n, 3), dtype=torch.float32, device=dev)
    buf_rew = torch.empty((RING, n), dtype=torch.float64, device=dev)
    buf_done = torch.empty((RING, n), dtype=torch.uint8, device=dev)
    buf_rstd = torch.zeros(RING, dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    row_offset = rank * n

    def full_step(t, tc=None):
        k = t % RING
        # pursuer and evader act on the same observation (CPPO_main.py:122-123): one launch for both networks on the tensor-core
        # path (the default), two FFMA2 launches at this batch size otherwise
        pursuer.sample_pair(evader, env=env, obs_stats=obs_stats, seed=11, step=2 * t, other_step=2 * t + 1, row_offset=row_offset,
                            act=buf_act[k], logp=buf_logp[k], obs_out=buf_obs[k], other_act=buf_eact[k], other_logp=buf_elogp[k], tc=tc)
        env.step(buf_act[k], buf_eact[k], reward=buf_rew[k], done=buf_done[k], obs_stats=obs_stats,
                 ret_stats=ret_stats, ret_std_out=buf_rstd[k:k + 1])

    # synthetic random actions, resident in HBM before the timed region (uniform in [-2, 2]: the clip is exercised)
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    rnd_pa = (torch.rand((RING, n, 3), generator=g, device=dev) * 4 - 2)
    rnd_ea = (torch.rand((RING, n, 3), generator=g, device=dev) * 4 - 2)

    def step(t):
        k = t % RING
        env.step(rnd_pa[k], rnd_ea[k], obs_f32=buf_obs[k], reward=buf_rew[k], done=buf_done[k], obs_stats=obs_stats,
                 ret_stats=ret_stats, ret_std_out=buf_rstd[k:k + 1])
    LAUNCHES_PER_STEP = 3   # env_front_rk4_kernel + env_step_kernel + stats_merge_kernel

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for t in range(args.warmup):
        step(t)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()                                               # evict L2 between timed steps
        ev[i][0].record()
        step(args.warmup + i)
        ev[i][1].record()
    barrier()
    wall = time.perf_counter() - wall0
    if args.dump_outputs and rank == 0:                             # before the sections below reuse the ring slots
        k = (args.warmup + args.steps - 1) % RING
        dump_outputs(args.dump_outputs, {"obs": buf_obs[k], "reward": buf_rew[k], "done": buf_done[k]},
                     {"ret_std": buf_rstd[k:k + 1]})
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    t_all = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    total_ms = float(t_all.item())
    ms_per_step = total_ms / args.steps
    value = n * world / (ms_per_step * 1e-3)

    # ---------------- per-kernel timings (each kernel alone, CUDA events on the launch stream)
    def time_kernel(fn, reps=10, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.mean(ts)), float(np.min(ts))

    # opt-in fast-libm variant of the same step (SatEnvParams.fast_libm: libdevice instead of the host libm's arithmetic in the
    # danger-zone count; not bit-identical to the reference there) on an identical second batch
    env_fast = eng.EnvBatch(n, mode="rk4", substeps=S, h=1.0, d_capture=20000.0, max_episode_steps=1000, auto_reset=True, device=dev,
                            fast_libm=True)
    env_fast.set_state(P, rng.normal(0, 3.0, (n, 3)), E, rng.normal(0, 3.0, (n, 3)))
    t_env_fast, _ = time_kernel(lambda: env_fast.step(rnd_pa[0], rnd_ea[0], obs_f32=buf_obs[0], reward=buf_rew[0], done=buf_done[0]))
    del env_fast
    k = 0
    t_env, t_env_min = time_kernel(lambda: env.step(rnd_pa[k], rnd_ea[k], obs_f32=buf_obs[k], reward=buf_rew[k], done=buf_done[k]))
    # per-launch split of the env step, CUDA events recorded between the launches on the launching stream
    split = []
    for _ in range(3):
        env.step_timed(rnd_pa[k], rnd_ea[k], reward=buf_rew[k], done=buf_done[k])
    for _ in range(10):
        flush.zero_()
        split.append(env.step_timed(rnd_pa[k], rnd_ea[k], reward=buf_rew[k], done=buf_done[k]))
    t_front, t_finish, t_merge = (float(np.mean([x[i] for x in split])) for i in range(3))
    cnt = [args.warmup + args.steps]
    def _full():
        full_step(cnt[0]); cnt[0] += 1
    t_full, t_full_min = time_kernel(_full)
    t_act, t_act_min = time_kernel(lambda: pursuer.sample(env=env, obs_stats=obs_stats, seed=11, step=0, act=buf_act[k], logp=buf_logp[k], tc=False))
    # the fp32 FFMA2 actors (csrc/actor.cu) in the same step, and the tensor-core kernel alone (one network / the pair)
    def _full_ff():
        full_step(cnt[0], tc=False); cnt[0] += 1
    t_full_ff, t_full_ff_min = time_kernel(_full_ff)
    t_act_tc, _ = time_kernel(lambda: pursuer.sample(env=env, obs_stats=obs_stats, seed=11, step=0, act=buf_act[k], logp=buf_logp[k], tc=True))
    t_pair_tc, _ = time_kernel(lambda: pursuer.sample_pair(evader, env=env, obs_stats=obs_stats, seed=11, step=0, other_step=1, act=buf_act[k],
                                                          logp=buf_logp[k], other_act=buf_eact[k], other_logp=buf_elogp[k], tc=True))
    # the same full step as 4 independent env shards ("virtual ranks": own running statistics, own stream) so that the
    # FP32 actor kernels of one shard overlap the FP64 env kernels of another
    def sharded_full_step_ms(parts_n=4, K=10):
        parts, streams = [], [torch.cuda.Stream(device=dev) for _ in range(parts_n)]
        m = n // parts_n
        for r_ in range(parts_n):
            e_ = eng.EnvBatch(m, mode="rk4", substeps=S, h=1.0, d_capture=20000.0, max_episode_steps=1000, device=dev)
            rr_ = np.random.default_rng(77 + r_)
            e_.set_state(np.array([200000.0, 0, 0]) + rr_.normal(0, 3e4, (m, 3)), rr_.normal(0, 3.0, (m, 3)),
                         np.array([18000.0, 0, 0]) + rr_.normal(0, 3e4, (m, 3)), rr_.normal(0, 3.0, (m, 3)))
            st_, rs_ = eng.RunningStats(18, dev), eng.RunningStats(1, dev)
            st_.update_normalize(e_.observe())
            parts.append((e_, st_, rs_, torch.zeros(1, dtype=torch.float64, device=dev)))

        def run(k0):
            cur = torch.cuda.current_stream(dev)
            for s_ in streams:
                s_.wait_stream(cur)
            for t_ in range(K):
                for r_, (e_, st_, rs_, sd_) in enumerate(parts):
                    lo_ = r_ * m
                    with torch.cuda.stream(streams[r_]):
                        pursuer.sample(env=e_, obs_stats=st_, seed=11, step=k0 + t_, row_offset=row_offset + lo_,
                                       act=buf_act[0, lo_:lo_ + m], logp=buf_logp[0, lo_:lo_ + m], obs_out=buf_obs[0, lo_:lo_ + m])
                        evader.sample(env=e_, obs_stats=st_, seed=12, step=k0 + t_, row_offset=row_offset + lo_,
                                      act=buf_eact[0, lo_:lo_ + m], logp=buf_elogp[0, lo_:lo_ + m])
                        e_.step(buf_act[0, lo_:lo_ + m], buf_eact[0, lo_:lo_ + m], reward=buf_rew[0, lo_:lo_ + m],
                                done=buf_done[0, lo_:lo_ + m], obs_stats=st_, ret_stats=rs_, ret_std_out=sd_)
            for s_ in streams:
                cur.wait_stream(s_)
        run(0)
        torch.cuda.synchronize()
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_.record(); run(K); b_.record(); b_.synchronize()
        return a_.elapsed_time(b_) / K
    t_full4 = sharded_full_step_ms() if n % 256 == 0 else None
    nk1 = 1 << 20
    xk1, _ = eng.alloc_soa(6, nk1, torch.float64, dev)
    ang = torch.rand(nk1, device=dev, dtype=torch.float64) * 6.283185307179586
    xk1[0], xk1[1], xk1[2] = 7000 * torch.cos(ang), 7000 * torch.sin(ang), 100 * torch.randn(nk1, device=dev, dtype=torch.float64)
    xk1[3], xk1[4], xk1[5] = -7.5 * torch.sin(ang), 7.5 * torch.cos(ang), 0.1 * torch.randn(nk1, device=dev, dtype=torch.float64)
    t_k1, t_k1_min = time_kernel(lambda: eng.rk4_propagate(xk1, 1.0, 100))
    # K4 + normalisation (SURVEY s8d: HBM-bound, 17 B/sample): GAE reverse scan, advantage moments + normalise, running-stats update
    def gae_case(T_, N_):
        r_ = torch.randn((T_, N_), device=dev); v_ = torch.randn((T_ + 1, N_), device=dev)
        d_ = (torch.rand((T_, N_), device=dev) < 0.02).to(torch.uint8)
        a_ = torch.empty_like(r_); vt_ = torch.empty_like(r_)
        ms, _ = time_kernel(lambda: eng.gae_time_major(r_, v_, d_, adv=a_, v_target=vt_), reps=5, warm=2)
        ms_m, _ = time_kernel(lambda: eng.adv_moments(a_), reps=5, warm=2)
        sums_ = eng.adv_moments(a_)
        ms_n, _ = time_kernel(lambda: eng.adv_normalize_(a_, sums=sums_, group=False), reps=5, warm=2)
        B_ = T_ * N_
        return {"T": T_, "N": N_, "gae_ms": ms, "gae_gbs": BYTES_GAE_SAMPLE * B_ / (ms * 1e-3) / 1e9,
                "adv_moments_ms": ms_m, "adv_moments_gbs": 4.0 * B_ / (ms_m * 1e-3) / 1e9,
                "adv_normalize_ms": ms_n, "adv_normalize_gbs": 8.0 * B_ / (ms_n * 1e-3) / 1e9}
    gae_cases = [gae_case(2048, 8192), gae_case(256, 65536)]
    xs_norm = torch.randn((65536, 18), dtype=torch.float64, device=dev)
    st_norm = eng.RunningStats(18, dev)
    t_norm, _ = time_kernel(lambda: st_norm.update_normalize(xs_norm, out_dtype=torch.float32), reps=5, warm=2)
    del xs_norm
    peak64 = eng.measure_vector_peak("fp64")
    peak32 = max(eng.measure_vector_peak("fp32"), eng.measure_vector_peak("fp32x2"))   # scalar FFMA vs packed FFMA2 chains
    ach_env = FLOP_ENV_STEP * (S / 100.0) * n / (t_env * 1e-3) / 1e12
    ach_k1 = FLOP_RK4_J2 * 100 * nk1 / (t_k1 * 1e-3) / 1e12
    ach_act = FLOP_ACTOR * n / (t_act * 1e-3) / 1e12

    # ---------------- e2e through the host-buffer API (pinned host actions in, obs/reward/done out)
    e2e = None
    if rank == 0 or world > 1:
        pa_h, ea_h, _o, _r, _d = env.host_buffers()                 # pinned host arrays: the step's inputs live there
        pa_h[...] = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        ea_h[...] = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        for _ in range(3):
            env.step_host(pa_h, ea_h)
        barrier()
        t0 = time.perf_counter()
        ke = max(5, min(args.steps, 20))
        for _ in range(ke):
            obs_h, rew_h, done_h = env.step_host(pa_h, ea_h)         # H2D actions, kernels, D2H obs/reward/done, sync
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": n * world * ke / float(dt.item()), "unit": "env-steps/s",
               "h2d_bytes_per_step": env.h2d_bytes_per_step, "d2h_bytes_per_step": env.d2h_bytes_per_step,
               "api": "EnvBatch.step_host(pa, ea) -> (obs, reward, done) = one sat_env_step_host call on pinned host arrays: the "
                      "propagation kernel reads the actions from host memory (zero-copy) and emits the next observation, a copy engine "
                      "moves it to the host on a second stream while the danger-zone kernel runs, reward/done are written to host "
                      "memory by that kernel; both streams are synchronised before the call returns; wall clock",
               "steps": ke, "rank_cpu_affinity": numa_cpus}
    # ---------------- BASELINE config 4: 1 048 576 envs sharded over the ranks (J2 on), on-device rollout of horizon 256
    config4 = None
    if (world > 1 or args.config4) and not args.no_config4:
        config4 = run_config4(args, rank, world, dev, torch, dist, eng)
    # ---------------- PPO samples/sec (BASELINE config 5 shape, per-GPU share): rollout + GAE + K-epoch update
    ppo = None
    if not args.no_ppo:
        ppo = run_ppo_section(args, rank, world, dev, torch, dist, eng)
        per_gpu_sample_steps = ppo["samples"] / world * 10
        ppo["optimizer_step_ms"] = 1e3 * ppo["update_s"] / ppo["optimizer_steps"]
        ppo["update_fp32_tflops_per_gpu"] = FLOP_PPO_SAMPLE_STEP * per_gpu_sample_steps / ppo["update_s"] / 1e12
        ppo["update_fp32_tflops_per_gpu_what"] = ("useful fp32 FLOPs of the update (827 392 per sample-step) per second; on the tensor-core path the "
                                                  "two 256-wide layer products and dW2 issue 6 bf16 word products per fp32 product, so this can exceed "
                                                  "the CUDA-core FFMA rate")
        ppo["update_frac_of_nominal_fp32_peak"] = ppo["update_fp32_tflops_per_gpu"] / FP32_NOMINAL_TFLOPS
        ppo["update_frac_of_measured_ffma_chain"] = ppo["update_fp32_tflops_per_gpu"] / peak32
        ppo["update_flops_per_sample_step"] = FLOP_PPO_SAMPLE_STEP
    clocks = sampler.stop() if rank == 0 else None     # sampled from warm-up to the end of every GPU-timed section

    if rank != 0:
        return
    # ---------------- CPU baseline on a bounded sample of the same workload (env step only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        probe, _ = cpu_env_steps_per_s(8 * cores, 1, S, cores)
        n_cpu = int(max(cores, min(n, probe * 2.0)))                 # ~2 s of CPU work per step ...
        k_cpu = int(max(2, min(50, round(12.0 * probe / n_cpu))))     # ... and ~12 s in total
        rate, dt = cpu_env_steps_per_s(n_cpu, k_cpu, S, cores)
        cpu = {"value": rate, "unit": "env-steps/s", "cores": cores, "kind": "port",
               "sample": f"{n_cpu} envs x {k_cpu} steps of the same env step (S={S} RK4+J2 substeps both craft + danger zone + reward), "
                         f"CPU oracle port in C with OpenMP on all {cores} host threads, {dt:.1f} s",
               # kind "reference": the reference's own Python on this host (BASELINE.md s3); these are different, much slower
               # workloads (single env, cw mode) and are reported beside the port, not used for the headline ratio
               "reference_python": reference_python_rows()}
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6650.0
    hbm_src = "MEASURED_PEAKS.json hbm_gbs" if os.path.exists(peaks_path) else "fallback 6650 GB/s (B200_PROFILING.md)"
    flop_step = FLOP_ENV_STEP * (S / 100.0)
    ach_front = flop_step * n / (t_front * 1e-3) / 1e12
    traffic_front, traffic_front_src = ncu_traffic("env_front_rk4_kernel", n)
    traffic_finish, traffic_finish_src = ncu_traffic("env_step_kernel", n)
    traffic_actor, traffic_actor_src = ncu_traffic("actor_tc_kernel_pair", n)
    if os.path.exists(peaks_path) and "bf16_tflops_sustained" in json.load(open(peaks_path)):
        bf16_peak, bf16_peak_src = json.load(open(peaks_path))["bf16_tflops_sustained"], "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a step)"
    else:
        bf16_peak, bf16_peak_src = 2250.0, "nominal dense bf16 2.25 PFLOP/s (no MEASURED_PEAKS.json)"
    for c in gae_cases:
        for k_ in ("gae", "adv_moments", "adv_normalize"):
            c[k_ + "_frac_of_hbm_peak"] = c[k_ + "_gbs"] / hbm_peak
    line = {
        "metric": "rk4_env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args, value),
        "rk4_steps_per_sec": value * 2 * S,
        "gpu_launches": LAUNCHES_PER_STEP * args.steps,
        "wall_s_timed_region": wall,
        "e2e": e2e,
        # FP64 / FP32 vector peaks are not in MEASURED_PEAKS.json: `peak` is the nominal pipe rate (lanes x 2 x max SM clock);
        # the FMA-chain microbenchmark of this run is reported beside it (frac_of_measured_chain)
        "roofline": {"kernel": "env_front_rk4_kernel: impulse + 2 x S RK4+J2 substeps of both craft = the dominant launch of the env step "
                               "and the one that performs all of the step's algorithmic (SURVEY s8d) FLOPs",
                     "bound": "fp64", "achieved": ach_front, "peak": FP64_NOMINAL_TFLOPS, "unit": "TFLOP/s",
                     "frac": ach_front / FP64_NOMINAL_TFLOPS,
                     "peak_source": "nominal FP64 pipe rate 148 SMs x 64 DFMA lanes x 2 x 1.965 GHz (MEASURED_PEAKS.json has no FP64 entry)",
                     "measured_dfma_chain_tflops": peak64, "frac_of_measured_chain": ach_front / peak64,
                     "launch_ms": t_front, "share_of_step": t_front / (t_front + t_finish + t_merge),
                     "traffic": traffic_front, "traffic_unit": "bytes per launch", "traffic_source": traffic_front_src,
                     "algorithmic_flops_per_env_step": flop_step, "algorithmic_bytes_per_env_step": BYTES_ENV_STEP,
                     "timing": "CUDA events recorded between the launches inside sat_env_step_timed, L2 flushed between iterations",
                     "whole_step": {"what": "front + finish (terminal checks, danger-zone root solves, reward, observations) + statistics "
                                            "merge, counting only the RK4 FLOPs as useful", "launch_ms": t_env, "launch_ms_min": t_env_min,
                                    "front_ms": t_front, "finish_ms": t_finish, "merge_ms": t_merge,
                                    "achieved": ach_env, "frac": ach_env / FP64_NOMINAL_TFLOPS,
                                    "finish_kernel_traffic": traffic_finish, "finish_kernel_traffic_source": traffic_finish_src,
                                    "hbm_achieved_gbs": BYTES_ENV_STEP * n / (t_env * 1e-3) / 1e9, "hbm_peak_gbs": hbm_peak}},
        # BASELINE config 3 exactly as worded ("full step ... with fused actor sampling"): both actors sample on the device, then the env step
        "config3_full_step": {
            "what": "pursuer + evader fused Gaussian actor sampling (observation rebuilt + normalised from the fp64 state, Philox "
                    "sampling, CPPO_main.py:122-123; both networks in ONE persistent tensor-core launch, sat_actor_sample_pair_tc) + the env "
                    "step above (:132); 5 launches (weight-image pack, actors, env front, env finish, statistics merge); CUDA events, L2 "
                    "flushed between steps",
            "ms_per_step": t_full, "ms_per_step_min": t_full_min, "per_gpu_env_steps_per_sec": n / (t_full * 1e-3),
            "env_steps_per_sec": n * world / (t_full * 1e-3),
            "split_ms": {"actor_pair": t_pair_tc, "env_front": t_front, "env_finish": t_finish, "stats_merge": t_merge},
            "roofline": {"kernel": "actor_tc_kernel (both dense layers of both actors as exact bf16x3 splits on tcgen05, accumulators in "
                                   "TMEM; %.0f %% of this step)" % (100 * t_pair_tc / t_full),
                         "bound": "tensor", "achieved": 6 * 2 * FLOP_ACTOR * n / (t_pair_tc * 1e-3) / 1e12, "peak": bf16_peak, "unit": "TFLOP/s",
                         "frac": 6 * 2 * FLOP_ACTOR * n / (t_pair_tc * 1e-3) / 1e12 / bf16_peak,
                         "peak_source": bf16_peak_src,
                         "what": "achieved = issued bf16 tensor FLOPs: 6 word products per fp32 product (exact 3-way split, 3 of 9 "
                                 "products dropped at 2^-24) x the actor's 141 824 fp32 FLOP per row x 2 networks; useful fp32 rate = "
                                 "achieved / 6",
                         "useful_fp32_tflops": 2 * FLOP_ACTOR * n / (t_pair_tc * 1e-3) / 1e12,
                         "launch_ms": t_pair_tc, "one_network_launch_ms": t_act_tc,
                         "traffic": traffic_actor, "traffic_source": traffic_actor_src},
            "ffma2_actor_variant": {
                "what": "the same full step with the fp32 CUDA-core actor kernels (actor_kernel<false>, FFMA2 register tiles; "
                        "GaussianActorKernel.sample(tc=False) / SAT_ACTOR_TC=0): two launches at this batch size. Accuracy against an "
                        "fp64 ground truth (tests/test_gpu_actor_tc.py): tensor-core path rms 6.5e-8 / FFMA2 7.2e-8 (tanh), 3.3e-8 / 3.5e-8 "
                        "(ReLU); same Philox stream",
                "ms_per_step": t_full_ff, "ms_per_step_min": t_full_ff_min, "per_gpu_env_steps_per_sec": n / (t_full_ff * 1e-3),
                "actor_launch_ms": t_act, "actor_fp32_tflops": ach_act, "actor_frac_of_nominal_fp32": ach_act / FP32_NOMINAL_TFLOPS,
                "tc_speedup_one_network": t_act / t_act_tc, "tc_speedup_pair": 2 * t_act / t_pair_tc},
            "as_4_independent_shards_on_4_streams": None if t_full4 is None else {
                "ms_per_step": t_full4, "per_gpu_env_steps_per_sec": n / (t_full4 * 1e-3),
                "what": "the same work as 4 env shards with per-shard running statistics on 4 streams: the FP32 actor kernels of "
                        "one shard overlap the FP64 env kernels of another"}},
        "config4": config4,
        "kernels": {
            "rk4_kernel (K1, 2^20 states x 100 substeps, J2)": {"ms": t_k1, "bound": "fp64", "achieved_tflops": ach_k1,
                                                              "frac_of_nominal_fp64_peak": ach_k1 / FP64_NOMINAL_TFLOPS,
                                                              "frac_of_measured_dfma_chain": ach_k1 / peak64,
                                                              "fp64_instr_per_rk4_step": FP64_INSTR_RK4_J2,
                                                              "fp64_pipe_busy_implied": (100 * nk1 / (t_k1 * 1e-3)) * FP64_INSTR_RK4_J2 / (FP64_NOMINAL_TFLOPS * 1e12 / 2),
                                                              "rk4_steps_per_sec": 100 * nk1 / (t_k1 * 1e-3)},
            "actor_kernel (K3, one actor)": {"ms": t_act, "bound": "fp32", "achieved_tflops": ach_act,
                                             "frac_of_nominal_fp32_peak": ach_act / FP32_NOMINAL_TFLOPS,
                                             "frac_of_measured_ffma_chain": ach_act / peak32},
            "env_step_kernel<rk4> (K2)": {"ms": t_env, "env_steps_per_sec": n / (t_env * 1e-3),
                                          "fast_libm_variant": {"ms": t_env_fast, "env_steps_per_sec": n / (t_env_fast * 1e-3),
                                                                "what": "SatEnvParams.fast_libm = 1 (opt-in): libdevice sin/cos/acos/atan and x*x in the "
                                                                        "danger-zone count instead of the host libm's own arithmetic; ~3e-5 of the integer "
                                                                        "counts then differ from the reference (round-1 behaviour). Default = exact"}},
            "gae + advantage normalisation (K4, bound hbm, 17 / 4 / 8 B per sample)": gae_cases,
            "sat_norm_update (65536 x 18 fp64 -> running stats + fp32 normalised)": {
                "ms": t_norm, "gbs": 65536 * 18 * (8 + 8 + 4) / (t_norm * 1e-3) / 1e9,
                "frac_of_hbm_peak": 65536 * 18 * (8 + 8 + 4) / (t_norm * 1e-3) / 1e9 / hbm_peak,
                "note": "4.7 MB per call: launch-latency bound (two passes + merge), not bandwidth bound"},
            "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src,
            "nominal_fp64_peak_tflops": FP64_NOMINAL_TFLOPS, "nominal_fp32_peak_tflops": FP32_NOMINAL_TFLOPS,
            "measured_dfma_chain_tflops": peak64, "measured_ffma_chain_tflops": peak32},
        "ppo": ppo,
        "cpu_baseline": cpu,
        "clocks": clocks,
    }
    emit(line)


_REAL_STDOUT = None


def emit(line):
    """the ONE JSON line goes to the real stdout; everything else (NCCL banners, warnings) was moved to stderr"""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                      # libraries that print to fd 1 (NCCL version banner) now land on stderr
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
