"""Statistics shared across ranks (sat_env_step_partials / sat_norm_partials / sat_stats_fold, EnvBatch.share_stats,
VectorTrainer(stats_group=...)): G shards that fold every shard's partials hold the statistics of the union batch, bit for
bit when every shard but the last holds a multiple of the rows per block, and a sharded rollout then equals the union
rollout. Emulated ranks in one process check the kernels and the C ABI; two processes on one GPU (gloo) and, where there
are two GPUs, two processes over NCCL check the exchange and the rollout."""
import os
import sys
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RESET_P, RESET_E = (200000.0, 0.0, 0.0), (18000.0, 0.0, 0.0)


def box(dp=50000.0, dv=3.0):
    c = np.array(RESET_P + (0.0, 0.0, 0.0) + RESET_E + (0.0, 0.0, 0.0))
    d = np.array([dp] * 3 + [dv] * 3 + [dp] * 3 + [dv] * 3)
    return c - d, c + d


def _eng():
    from ppo_rl_satellite_b200 import engine
    return engine


def _env(eng, n, mode, row_offset=0, device="cuda"):
    return eng.EnvBatch(n, mode=mode, d_capture=20000.0, max_episode_steps=12, start_box=box(), start_seed=21,
                        row_offset=row_offset, device=device)


def _norm_fold(eng, xs, stats):
    """sat_norm_partials of every shard xs[k], gathered rank-major, folded into each stats[k]"""
    lib = eng.L.load()
    dim = xs[0].shape[1]
    rows = [x.shape[0] for x in xs]
    stride = max(lib.sat_stats_partials_bytes(m, dim) for m in rows) // 8
    ws = torch.zeros(eng.L.load().sat_workspace_bytes(1), dtype=torch.uint8, device="cuda")
    sends = []
    for x in xs:
        send = torch.zeros(stride, dtype=torch.float64, device="cuda")
        eng.L.check(lib.sat_norm_partials(eng.L.ptr(x), x.shape[0], dim, eng.L.ptr(send), ws.data_ptr(),
                                          eng.L.stream_ptr()), "sat_norm_partials")
        sends.append(send)
    gathered = torch.stack(sends)
    rank_rows = torch.tensor(rows, dtype=torch.int64, device="cuda")
    for st in stats:
        eng.fold_stats(gathered, rank_rows, dim, st, workspace=ws)


def _run_shards(mode, sizes, steps, exact):
    """G shards (rank_rows = sizes) against one batch of the union stepping the same global actions, and (exact) a union
    batch whose own partials go through the fold as one rank, against sat_env_step / sat_norm_update's merge"""
    eng = _eng()
    lib = eng.L.load()
    N, G = sum(sizes), len(sizes)
    offs = np.cumsum((0,) + tuple(sizes))
    U = _env(eng, N, mode)
    U1 = _env(eng, N, mode)
    S = [_env(eng, m, mode, row_offset=int(o)) for m, o in zip(sizes, offs[:-1])]
    new = lambda: (eng.RunningStats(18), eng.RunningStats(1), torch.zeros(1, dtype=torch.float64, device="cuda"))
    u, u1, s = new(), new(), [new() for _ in S]

    # the initial observations (RunningStats.update_normalize's path)
    u[0].update_normalize(U.observe())
    _norm_fold(eng, [U1.observe()], [u1[0]])
    _norm_fold(eng, [e.observe() for e in S], [x[0] for x in s])

    def check_stats(t):
        ref = torch.cat([u[0].buf, u[1].buf, u[2]])
        got = [torch.cat([x[0].buf, x[1].buf, x[2]]) for x in s]
        for k in range(1, G):
            assert torch.equal(got[k], got[0]), f"step {t}: shard {k}'s statistics differ from shard 0's"
        if exact:
            assert torch.equal(torch.cat([u1[0].buf, u1[1].buf, u1[2]]), ref), f"step {t}: G = 1 fold != sat_env_step"
            for k in range(G):
                assert torch.equal(got[k], ref), f"step {t}: shard {k}'s statistics differ from the union's"
        else:
            for st, ust in ((s[0][0], u[0]), (s[0][1], u[1])):
                assert st.n == ust.n
                d = st.dim
                a, b = st.buf.cpu().numpy(), ust.buf.cpu().numpy()
                sd = b[1 + 2 * d:1 + 3 * d]
                assert np.all(np.abs(a[1:1 + d] - b[1:1 + d]) <= 1e-12 * (np.abs(b[1:1 + d]) + sd)), f"step {t}: mean"
                assert np.all(np.abs(a[1 + d:] - b[1 + d:]) <= 1e-12 * np.abs(b[1 + d:])), f"step {t}: S / std"

    check_stats(-1)
    stride = max(lib.sat_stats_partials_bytes(m, 0) for m in sizes) // 8
    sends = [torch.zeros(stride, dtype=torch.float64, device="cuda") for _ in S]
    p1 = torch.zeros(1, lib.sat_stats_partials_bytes(N, 0) // 8, dtype=torch.float64, device="cuda")
    rank_rows = torch.tensor(sizes, dtype=torch.int64, device="cuda")
    rows1 = torch.tensor([N], dtype=torch.int64, device="cuda")
    uobs, u1obs = (torch.empty((N, 18), dtype=torch.float64, device="cuda") for _ in range(2))
    sobs = [torch.empty((m, 18), dtype=torch.float64, device="cuda") for m in sizes]
    resets = 0
    for t in range(steps):
        g = torch.Generator(device="cuda").manual_seed(1000 + t)
        pa = torch.rand((N, 3), generator=g, device="cuda", dtype=torch.float32) * 4 - 2
        ea = torch.rand((N, 3), generator=g, device="cuda", dtype=torch.float32) * 4 - 2
        U.step(pa, ea, obs_f64=uobs, obs_stats=u[0], ret_stats=u[1], ret_std_out=u[2])
        if exact:
            U1.step_partials(pa, ea, p1, obs_f64=u1obs)
            eng.fold_stats(p1, rows1, 0, u1[0], u1[1], u1[2], U1.workspace)
        for k, e in enumerate(S):
            e.step_partials(pa[offs[k]:offs[k + 1]], ea[offs[k]:offs[k + 1]], sends[k], obs_f64=sobs[k])
        gathered = torch.stack(sends)
        for k, e in enumerate(S):
            eng.fold_stats(gathered, rank_rows, 0, s[k][0], s[k][1], s[k][2], e.workspace)
        for k, e in enumerate(S):
            lo, hi = offs[k], offs[k + 1]
            assert torch.equal(sobs[k], uobs[lo:hi]) and torch.equal(e.reward, U.reward[lo:hi]), f"step {t} shard {k}"
            assert torch.equal(e.done, U.done[lo:hi]), f"step {t} shard {k}"
        resets += int(U.done.sum())
        check_stats(t)
    assert resets > N                                  # every env finished at least one episode on average
    return u


@pytest.mark.parametrize("mode", ["cw", "rk4"])
@pytest.mark.parametrize("sizes", [(4096,) * 4, (8192, 4133), (4096, 4096, 4096, 37)],
                         ids=["4x4096", "8192|4133", "3x4096|37"])
def test_emulated_ranks_fold_to_the_bits_of_the_union(mode, sizes):
    _run_shards(mode, sizes, 56, exact=True)


def test_misaligned_interior_shard_agrees_to_rounding():
    """an interior shard of 4101 rows cuts the blocks elsewhere than the union: every shard still holds the same bits, and
    they agree with the union's statistics to 1e-12 relative"""
    _run_shards("cw", (4096 + 5, 4091), 24, exact=False)


# ------------------------------------------------------------------------------------------------ rollout, 2 ranks
N_UNION, T = 2 * 4096, 64


def _args(B, mb):
    return types.SimpleNamespace(policy_dist="Gaussian", max_action=1.6, batch_size=B, mini_batch_size=mb, max_train_steps=int(3e6),
                                 lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1, K_epochs=1, entropy_coef=0.01,
                                 set_adam_eps=True, use_grad_clip=True, use_lr_decay=True, use_adv_norm=False, state_dim=18,
                                 action_dim=3, hidden_width=256, use_tanh=1, use_orthogonal_init=True, chkpt_dir="/tmp")


def _agents(n, T_, device):
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    torch.manual_seed(0)
    a = P.PPO_continuous(_args(n * T_, 2048), "pursuer", device=device)
    b = P.PPO_continuous(_args(n * T_, 2048), "evader", device=device)
    with torch.no_grad():                      # make the policy means matter
        for m in (a, b):
            m.actor.mean_layer.weight.mul_(30.0)
    a._dirty = b._dirty = True
    return a, b


def _rollout(n, rank, device, group):
    eng = _eng()
    from ppo_rl_satellite_b200 import rollout
    env = _env(eng, n, "cw", row_offset=rank * n, device=device)
    agent, opp = _agents(n, T, device)
    tr = rollout.VectorTrainer(env, agent, opp, T, rank=rank, seed=5, stats_group=group)
    tr.collect()
    tr.compute_advantages(group=group)
    b = tr.buf
    out = {k: getattr(b, k).cpu().numpy() for k in ("obs", "act", "logp", "opp_act", "opp_logp", "rew64", "done", "ret_std",
                                                   "values", "adv", "v_target")}
    out["obs_stats"], out["ret_stats"] = tr.obs_stats.buf.cpu().numpy(), tr.ret_stats.buf.cpu().numpy()
    return out


def _selfplay_stats(n, rank, device, group):
    eng = _eng()
    from ppo_rl_satellite_b200 import rollout
    env = _env(eng, n, "cw", row_offset=rank * n, device=device)
    sp = rollout.SelfPlay(env, *_agents(n, 8, device), 8, 2048, rank=rank, seed=9, stats_group=group)
    sp.run_phase(0, 1, group=group)
    tr = sp.trainers[0]
    return np.concatenate([tr.obs_stats.buf.cpu().numpy(), tr.ret_stats.buf.cpu().numpy()])


def _rank_worker(rank, world, port, backend, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world, **({"device_id": dev} if backend == "nccl" else {}))
    try:
        res = _rollout(N_UNION // world, rank, dev, dist.group.WORLD)
        res["selfplay"] = _selfplay_stats(N_UNION // world, rank, dev, dist.group.WORLD)
        torch.cuda.synchronize()
        q.put((rank, res))
    except BaseException as exc:
        q.put((rank, repr(exc)))
        raise
    finally:
        dist.destroy_process_group()


def _check_two_ranks(backend, port_base):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = port_base + (os.getpid() % 2000)
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, backend, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=400) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for r in range(2):
        assert isinstance(res[r], dict), f"rank {r} failed: {res[r]}"
    one = _rollout(N_UNION, 0, torch.device("cuda", 0), None)
    n = N_UNION // 2
    for r in range(2):
        for k in ("obs", "act", "logp", "opp_act", "opp_logp", "rew64", "done", "values", "adv", "v_target"):
            assert np.array_equal(res[r][k], one[k][:, r * n:(r + 1) * n]), f"rank {r}: {k} differs from the union's slice"
        for k in ("ret_std", "obs_stats", "ret_stats"):
            assert np.array_equal(res[r][k], one[k]), f"rank {r}: {k} differs from the union's"
    assert np.array_equal(res[0]["selfplay"], res[1]["selfplay"])
    assert res[0]["selfplay"][0] > 0


@pytest.mark.timeout(600)
def test_two_ranks_one_gpu_gloo_rollout_equals_the_union_rollout():
    _check_two_ranks("gloo", 31100)


@pytest.mark.timeout(600)
def test_two_gpus_nccl_rollout_equals_the_union_rollout():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _check_two_ranks("nccl", 33300)
