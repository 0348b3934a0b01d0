import os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppo_rl_satellite_b200 import engine as eng
n = 65536
env = eng.EnvBatch(n, mode="rk4", substeps=100, h=1.0, d_capture=20000.0, max_episode_steps=1000)
pa, ea, obs, rew, done = env.host_buffers()
rng = np.random.default_rng(0)
pa[...] = rng.uniform(-2, 2, (n, 3)); ea[...] = rng.uniform(-2, 2, (n, 3))
for _ in range(3): env.step_host(pa, ea)
torch.cuda.synchronize(); t0 = time.perf_counter()
for _ in range(20): env.step_host(pa, ea)
dt = (time.perf_counter() - t0) / 20
print(f"step_host: {dt*1e6:.0f} us/step -> {n/dt:.3e} env-steps/s")
# raw copies
d = torch.empty((n, 18), dtype=torch.float32, device="cuda"); h = torch.empty((n, 18), dtype=torch.float32).pin_memory()
for name, fn in (("D2H 4.7MB", lambda: h.copy_(d, non_blocking=True)), ("H2D 4.7MB", lambda: d.copy_(h, non_blocking=True))):
    for _ in range(3): fn()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(20): fn()
    torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / 20
    print(f"{name}: {dt*1e6:.0f} us -> {h.numel()*4/dt/1e9:.1f} GB/s")
