"""Host restatements of the reference's advantage block (ppo_continuous.py:198-210) used by the GAE tests.

reference_block: the block itself, line for line, as it runs under numpy 2 (SURVEY H4): the deltas are torch CPU fp32
tensor operations, the recursion runs over np.float32 scalars, and gamma * lamda is a python float product that NEP 50
casts to float32 only when it meets the np.float32 gae.

gae_scan: the same arithmetic for a time-major [T, N] rollout, vectorised across the env columns, in the CUDA kernel's
operation order: delta = (r + (f32(gamma) (1 - d)) v') - v, then g = delta + (f32(gamma lamda) (1 - d)) g. Every numpy
operation here is one correctly rounded fp32 operation, so it is an exact reference for the kernel.

gae_fp64: the recursion in fp64 with gl = gamma lamda, an independent check of gae_scan within a rounding bound."""
import numpy as np

F32 = np.float32


def reference_block(r, vs, vs_, dw, done, gamma, lamda):
    """ppo_continuous.py:198-208 on (B, 1) buffers of one env in time order; returns (adv, v_target) as flat float32"""
    import torch
    r, vs, vs_, dw, done = (torch.from_numpy(np.ascontiguousarray(a, dtype=F32).reshape(-1, 1))
                            for a in (r, vs, vs_, dw, done))
    adv = []
    gae = 0
    with torch.no_grad():
        deltas = r + gamma * (1.0 - dw) * vs_ - vs
        for delta, d in zip(reversed(deltas.flatten().numpy()), reversed(done.flatten().numpy())):
            gae = delta + gamma * lamda * gae * (1.0 - d)
            adv.insert(0, gae)
        adv = torch.tensor(adv, dtype=torch.float).view(-1, 1)
        v_target = adv + vs
    return adv.numpy().ravel(), v_target.numpy().ravel()


def scaled_rewards(r, r_scale=None):
    """r * r_scale[t] in fp32, as the kernel applies the per-step reward scale"""
    r = np.asarray(r, dtype=F32)
    return r if r_scale is None else r * np.asarray(r_scale, dtype=F32)[:, None]


def gae_scan(r, v, done, gamma, lamda, r_scale=None):
    """r, done [T, N]; v [T+1, N]; r_scale [T] or None. Returns (adv, v_target) [T, N] float32."""
    r = scaled_rewards(r, r_scale)
    v = np.asarray(v, dtype=F32)
    keep = F32(1.0) - (np.asarray(done) != 0).astype(F32)
    delta = (r + (F32(gamma) * keep) * v[1:]) - v[:-1]
    coef = F32(gamma * lamda) * keep
    adv = np.empty_like(r)
    g = np.zeros(r.shape[1], dtype=F32)
    for t in range(r.shape[0] - 1, -1, -1):
        g = delta[t] + coef[t] * g
        adv[t] = g
    return adv, adv + v[:-1]


def gae_fp64(r, v, done, gamma, lamda, r_scale=None):
    """fp64 GAE of the same fp32 inputs (rewards scaled in fp32 first, as the kernel does). Returns (adv, delta) fp64."""
    r = scaled_rewards(r, r_scale).astype(np.float64)
    v = np.asarray(v, dtype=np.float64)
    keep = 1.0 - (np.asarray(done) != 0)
    delta = r + gamma * keep * v[1:] - v[:-1]
    adv = np.empty_like(r)
    g = np.zeros(r.shape[1])
    for t in range(r.shape[0] - 1, -1, -1):
        g = delta[t] + gamma * lamda * keep[t] * g
        adv[t] = g
    return adv, delta
