"""Cost of starts mode (EnvBatch(start_box=...)) on the env step: default-mode and starts-mode steps of the same size,
alternated on the same seeded actions, CUDA events around each step, L2 flushed before each one.

    python tools/time_env_starts.py [--envs 65536] [--steps 40] [--warmup 5] [--max-episode-steps 20]

cw mode and rk4 mode (S = 100 substeps of 1 s, J2 on). All batches start from the same states; the default batch then
resets to the reference's literals and the starts batch to its drawn starts; the episode counters start staggered, so
about 1/max_episode_steps of the envs reset on every step. A starts-mode EnvBatch.step is the step launches plus the
sat_env_draw_starts launch for the envs the step finished. A third batch, "fixed", runs starts mode with lo == hi == the
reference's reset literals: the starts-mode kernels on the default batch's workload (its resets land on the same
geometry), which separates the cost of the code from the cost of resetting to varied geometries (the danger-zone solve
of the reference's reset geometry is cheaper than that of a random one). Three timings per mode, each rotating the
order of the batches from step to step:
  step     EnvBatch.step (events around it: every launch of the call, incl. the draw in starts mode)
  kernels  the step's launches alone (sat_env_step_timed: front + finish + statistics merge), no draw
  draw     the draw launch alone, on a mask with 1/max_episode_steps of the rows set and on all rows
The step carries the observation / return statistics, as in VectorTrainer. Prints the card name and power limit, the
per-mode times, and one JSON line. Writes nothing."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppo_rl_satellite_b200 import engine as eng  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def box():
    c = np.array([200000.0, 0, 0, 0, 0, 0, 18000.0, 0, 0, 0, 0, 0])
    d = np.array([50000.0] * 3 + [3.0] * 3 + [50000.0] * 3 + [3.0] * 3)
    return c - d, c + d


def run_mode(mode, n, steps, warmup, max_steps):
    kw = dict(mode=mode, d_capture=20000.0, max_episode_steps=max_steps)
    if mode == "rk4":
        kw.update(substeps=100, h=1.0)
    starts = eng.EnvBatch(n, start_box=box(), start_seed=1, **kw)
    default = eng.EnvBatch(n, **kw)
    lit = np.array([200000.0, 0, 0, 0, 0, 0, 18000.0, 0, 0, 0, 0, 0])
    fixed = eng.EnvBatch(n, start_box=(lit, lit), **kw)
    s0 = starts.state[:12].cpu().numpy()
    count0 = torch.arange(n, device="cuda", dtype=torch.int32) % max_steps
    for env in (starts, default, fixed):
        if env is not starts:
            env.set_state(s0[0:3].T, s0[3:6].T, s0[6:9].T, s0[9:12].T)
        env.episode_count.copy_(count0)
    g = torch.Generator(device="cuda").manual_seed(99)
    acts = [(torch.rand((n, 3), generator=g, device="cuda") * 4 - 2, torch.rand((n, 3), generator=g, device="cuda") * 4 - 2)
            for _ in range(8)]
    io = {}
    names = ("default", "starts", "fixed")
    order = lambda i: names[i % 3:] + names[:i % 3]
    for name, env in zip(names, (default, starts, fixed)):
        io[name] = dict(env=env, obs=torch.empty((n, 18), dtype=torch.float32, device="cuda"),
                        st=eng.RunningStats(18), rs=eng.RunningStats(1), ms=[], kms=[], resets=0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for i in range(warmup + steps):
        pa, ea = acts[i % 8]
        for name in order(i):
            b = io[name]
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _, d = b["env"].step(pa, ea, obs_f32=b["obs"], obs_stats=b["st"], ret_stats=b["rs"])
            e1.record()
            e1.synchronize()
            if i >= warmup:
                b["ms"].append(e0.elapsed_time(e1))
                b["resets"] += int(d.sum())
    for i in range(warmup + steps):
        pa, ea = acts[i % 8]
        for name in order(i):
            b = io[name]
            flush.zero_()
            torch.cuda.synchronize()
            ms = b["env"].step_timed(pa, ea, obs_stats=b["st"], ret_stats=b["rs"])
            if i >= warmup:
                b["kms"].append(sum(ms))
    # the draw launch alone (its own draw indices: the batch is not stepped afterwards)
    g2 = torch.Generator(device="cuda").manual_seed(5)
    masks = {"draw_part": (torch.rand(n, generator=g2, device="cuda") < 1.0 / max_steps).to(torch.uint8),
             "draw_all": torch.ones(n, dtype=torch.uint8, device="cuda")}
    draw = {}
    for key, mask in masks.items():
        for _ in range(5):
            starts.draw_starts(mask)
        t = []
        for _ in range(50):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); starts.draw_starts(mask); e1.record(); e1.synchronize()
            t.append(e0.elapsed_time(e1))
        draw[key] = (float(np.median(t)), int(mask.sum()))
    res = {"mode": mode, "envs": n, "steps": steps, "max_episode_steps": max_steps}
    for name in names:
        ms = np.array(io[name]["ms"])
        res[f"{name}_ms_mean"] = float(ms.mean())
        res[f"{name}_ms_median"] = float(np.median(ms))
        res[f"{name}_ms_std"] = float(ms.std())
        res[f"{name}_kernels_ms_median"] = float(np.median(io[name]["kms"]))
        res[f"{name}_resets_per_step"] = io[name]["resets"] / steps / n
    res["starts_over_default"] = res["starts_ms_median"] / res["default_ms_median"]
    res["starts_kernels_over_default"] = res["starts_kernels_ms_median"] / res["default_kernels_ms_median"]
    res["fixed_over_default"] = res["fixed_ms_median"] / res["default_ms_median"]
    res["fixed_kernels_over_default"] = res["fixed_kernels_ms_median"] / res["default_kernels_ms_median"]
    for key, (t, rows) in draw.items():
        res[f"{key}_ms_median"], res[f"{key}_rows"] = t, rows
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--max-episode-steps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_env_starts.py needs a CUDA device")
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}")
    out = {"card": name, "power_limit_and_max_sm_clock": power, "results": []}
    for mode in ("cw", "rk4"):
        r = run_mode(mode, a.envs, a.steps, a.warmup, a.max_episode_steps)
        out["results"].append(r)
        print(f"{mode:>3}: {r['envs']} envs, {r['starts_resets_per_step']:.3f} of the envs reset per step (default "
              f"{r['default_resets_per_step']:.3f}). Medians: step default {r['default_ms_median'] * 1e3:.1f} us, starts "
              f"{r['starts_ms_median'] * 1e3:.1f} us (x{r['starts_over_default']:.3f}); step kernels alone default "
              f"{r['default_kernels_ms_median'] * 1e3:.1f} us, starts {r['starts_kernels_ms_median'] * 1e3:.1f} us "
              f"(x{r['starts_kernels_over_default']:.3f}); fixed box (reference literals): step "
              f"{r['fixed_ms_median'] * 1e3:.1f} us (x{r['fixed_over_default']:.3f}), kernels "
              f"{r['fixed_kernels_ms_median'] * 1e3:.1f} us (x{r['fixed_kernels_over_default']:.3f}); draw launch alone {r['draw_part_ms_median'] * 1e3:.1f} us "
              f"({r['draw_part_rows']} rows), {r['draw_all_ms_median'] * 1e3:.1f} us ({r['draw_all_rows']} rows)")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
