"""PPO optimiser step at minibatch mb: fused CUDA kernels vs the CUDA-graphed PyTorch step

    python tools/time_ppo_fused.py [mb,mb,...]      # fused vs graphed PyTorch step
    python tools/time_ppo_fused.py --stats [rounds] # fused step with training diagnostics off / off again / on, alternated
"""
import os, subprocess, sys, time
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from ppo_rl_satellite_b200.dropin import ppo_continuous as P

argv = [x for x in sys.argv[1:] if x != "--stats"]
B = 1 << 21
a = bench._PpoArgs(policy_dist="Gaussian", max_action=1.6, batch_size=B, mini_batch_size=65536, max_train_steps=int(3e6),
                   lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1, K_epochs=1, entropy_coef=0.01, set_adam_eps=True,
                   use_grad_clip=True, use_lr_decay=True, use_adv_norm=True, state_dim=18, action_dim=3, hidden_width=256,
                   use_tanh=True, use_orthogonal_init=True, chkpt_dir="/tmp")
s = torch.randn(B, 18, device="cuda"); act = torch.randn(B, 3, device="cuda").clamp(-1.6, 1.6); lp = torch.randn(B, 3, device="cuda") * 0.1 - 1.0
adv = torch.randn(B, 1, device="cuda"); vt = torch.randn(B, 1, device="cuda")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or f"{torch.cuda.get_device_name()}, power limit unknown"


def time_step(agent, mb, **kw):
    """ms per optimiser step over one epoch of B rows (device events)"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); agent.optimize(s, act, lp, adv, vt, mini_batch_size=mb, **kw); e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) / -(-B // mb)


if "--stats" in sys.argv:
    # The same agent runs every mode so that the weights, workspace and streams are shared; the order rotates each round so
    # that drift of the shared machine does not favour one mode. "off2" is stats off again: its distance from "off" is the
    # run-to-run noise against which the stats-on overhead is read.
    rounds = int(argv[0]) if argv else 20
    print(f"card: {card()}")
    for mb in (65536, 148 * 128 * 2 + 37):
        agent = P.PPO_continuous(a, "pursuer")
        modes = {"off": dict(fused=True), "off2": dict(fused=True), "on": dict(fused=True, stats=True)}
        for kw in modes.values():
            agent.optimize(s, act, lp, adv, vt, mini_batch_size=mb, **kw)
        torch.cuda.synchronize()
        t = {k: [] for k in modes}
        names = list(modes)
        for r in range(rounds):
            for k in names[r % 3:] + names[:r % 3]:
                t[k].append(time_step(agent, mb, **modes[k]))
        med = {k: sorted(v)[len(v) // 2] for k, v in t.items()}
        print(f"mb {mb}: ms per optimiser step (median of {rounds}, {-(-B // mb)} steps each): "
              + ", ".join(f"{k} {med[k]:.4f} (min {min(t[k]):.4f})" for k in names)
              + f"; off2 - off {1e3 * (med['off2'] - med['off']):+.1f} us, on - off {1e3 * (med['on'] - med['off']):+.1f} us "
              f"({100 * (med['on'] / med['off'] - 1):+.2f} %)")
    sys.exit(0)

mbs = [int(x) for x in (argv[0].split(",") if argv else ["65536", "75776"])]
for mb in mbs:
    for mode in ("fused", "graph"):
        agent = P.PPO_continuous(a, "pursuer")
        kw = dict(fused=True) if mode == "fused" else dict(use_graph=True)
        agent.optimize(s, act, lp, adv, vt, mini_batch_size=mb, **kw)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(); agent.optimize(s, act, lp, adv, vt, mini_batch_size=mb, **kw); e1.record(); e1.synchronize()
        steps = -(-B // mb)
        print(f"mb {mb} {mode}: {e0.elapsed_time(e1) / steps:.3f} ms per optimiser step ({steps} steps, host {1e3 * (time.perf_counter() - t0) / steps:.3f} ms), "
              f"{B / (e0.elapsed_time(e1) * 1e-3):.3e} samples/s/epoch")
