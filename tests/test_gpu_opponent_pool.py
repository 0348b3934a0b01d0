"""Opponent pool (csrc/actor_tc.cu pool launch, sat_actor_tc_snapshot / sat_actor_sample_pool_tc, engine.OpponentPool,
GaussianActorKernel.sample_vs_pool, VectorTrainer / SelfPlay opponent_pool): the learner and K frozen snapshots, each on its
own group of rows, in one tensor-core launch, bit for bit the learner's pair-launch outputs and each snapshot's own
sat_actor_sample_tc on its rows."""
import copy
import ctypes as C
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

RESET_P, RESET_E = (200000.0, 0.0, 0.0), (18000.0, 0.0, 0.0)


@pytest.fixture(scope="module")
def eng():
    from ppo_rl_satellite_b200 import engine
    return engine


def _weights(seed):
    import bench
    W = {k: v.numpy().copy() for k, v in bench.orthogonal_actor_state(torch, seed).items()}
    rng = np.random.default_rng(seed)
    W["fc1.bias"] = rng.normal(0, 0.1, 256).astype(np.float32)
    W["fc2.bias"] = rng.normal(0, 0.1, 256).astype(np.float32)
    W["mean_layer.weight"] = (W["mean_layer.weight"] * 20.0).astype(np.float32)     # make the means differ between nets
    W["mean_layer.bias"] = rng.normal(0, 0.1, 3).astype(np.float32)
    W["log_std"] = rng.normal(-0.3, 0.2, (1, 3)).astype(np.float32)
    return W


def _kernel(eng, seed, use_tanh=True):
    return eng.GaussianActorKernel(use_tanh=use_tanh).load_state_dict(_weights(seed))


def _pool(eng, K, use_tanh=True, seed0=100):
    pool = eng.OpponentPool(K, use_tanh=use_tanh)
    for k in range(K):
        pool.add(_kernel(eng, seed0 + k, use_tanh))
    return pool


def _random_env(eng, n, seed):
    rng = np.random.default_rng(seed)
    env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=10)
    P = np.array(RESET_P) + rng.normal(0, 3e4, (n, 3)); E = np.array(RESET_E) + rng.normal(0, 3e4, (n, 3))
    env.set_state(P, rng.normal(0, 3.0, (n, 3)), E, rng.normal(0, 3.0, (n, 3)))
    st = eng.RunningStats(18)
    st.update_normalize(env.observe())
    return env, st


def _sub_state(L, env, lo, hi):
    """the env-state view of rows [lo, hi) (same column stride)"""
    return L.SatEnvState(env._state_buf.data_ptr() + 8 * lo, env._istate_buf.data_ptr() + 4 * lo, hi - lo, env.ld)


def _outs(n, k=5):
    return [torch.full((n, 3), float("nan"), dtype=torch.float32, device="cuda") for _ in range(k)]


@pytest.mark.timeout(600)
@pytest.mark.parametrize("use_tanh", [True, False])
@pytest.mark.parametrize("K", [1, 3, 8, 16])
@pytest.mark.parametrize("size", ["one_tile_per_group", 8192, 65536 + 37])
def test_pool_launch_equals_reference(eng, use_tanh, K, size):
    from ppo_rl_satellite_b200 import rollout
    L = eng.L
    lib = L.load()
    n = 128 * K if size == "one_tile_per_group" else size
    ends = rollout.pool_group_bounds(n, K)
    assert all(b > a for a, b in zip([0] + ends, ends))
    learner = _kernel(eng, 1, use_tanh)
    pool = _pool(eng, K, use_tanh)
    slots = list(range(K))[::-1]                               # group k plays slot K - 1 - k
    seed, step, other_step, R = 0x1234_5678_9abc, 10, 11, 3 * 65536
    m64 = 2 ** 64 - 1

    # fp32 observations
    x = torch.from_numpy(np.random.default_rng(K).normal(0, 1.5, (n, 18)).astype(np.float32)).cuda()
    a, lp, oa, olp = _outs(n, 4)
    obs_out = torch.full((n, 18), float("nan"), dtype=torch.float32, device="cuda")
    learner.sample_vs_pool(pool, slots, ends, obs=x, seed=seed, step=step, other_step=other_step, row_offset=R, act=a,
                           logp=lp, obs_out=obs_out, other_act=oa, other_logp=olp, tc=True)
    ra, rlp, _, _ = learner.sample_pair(pool.kernel(0), obs=x, seed=seed, step=step, other_step=other_step, row_offset=R,
                                        tc=True)
    assert torch.equal(a, ra) and torch.equal(lp, rlp) and torch.equal(obs_out, x)
    lo = 0
    for s, e in zip(slots, ends):
        ga, glp = pool.kernel(s).sample(obs=x[lo:e].contiguous(), seed=seed, step=other_step, row_offset=R + lo, tc=True)
        assert torch.equal(oa[lo:e], ga) and torch.equal(olp[lo:e], glp), f"group ending at {e} (slot {s})"
        lo = e

    # the env-state path: observation rebuilt and normalised inside the kernel (C ABI)
    env, st = _random_env(eng, n, K)
    a, lp, oa, olp, _ = _outs(n)
    o1 = torch.full((n, 18), float("nan"), dtype=torch.float32, device="cuda"); o2 = torch.empty_like(o1)
    arr = (L.SatActorPoolGroup * K)()
    for k, (s, e) in enumerate(zip(slots, ends)):
        arr[k] = pool.group(s)
        arr[k].row_end = e
    L.check(lib.sat_actor_sample_pool_tc(C.byref(learner.w), learner._image().data_ptr(), arr, K, None, C.byref(env.st),
                                         L.ptr(st.buf), n, R, seed & m64, step, other_step, L.ptr(a), L.ptr(lp), L.ptr(o1),
                                         L.ptr(oa), L.ptr(olp), L.stream_ptr()), "pool")
    ra, rlp, rb, rblp = _outs(n, 4)
    other = pool.kernel(0)
    other_img = torch.empty(L.ACTOR_TC_IMAGE_FLOATS, dtype=torch.float32, device="cuda")
    L.check(lib.sat_actor_sample_pair_tc(C.byref(learner.w), C.byref(other.w), learner._image().data_ptr(),
                                         other_img.data_ptr(), None, C.byref(env.st), L.ptr(st.buf), n, R, seed & m64, step,
                                         other_step, L.ptr(ra), L.ptr(rlp), L.ptr(o2), L.ptr(rb), L.ptr(rblp),
                                         L.stream_ptr()), "pair")
    assert torch.equal(a, ra) and torch.equal(lp, rlp) and torch.equal(o1, o2)
    lo = 0
    for s, e in zip(slots, ends):
        ga, glp = _outs(e - lo, 2)
        sub = _sub_state(L, env, lo, e)
        k = pool.kernel(s)
        L.check(lib.sat_actor_sample_tc(C.byref(k.w), k._image().data_ptr(), None, C.byref(sub), L.ptr(st.buf), e - lo,
                                        R + lo, seed & m64, other_step, None, L.ptr(ga), L.ptr(glp), None, None, None,
                                        L.stream_ptr()), "single")
        assert torch.equal(oa[lo:e], ga) and torch.equal(olp[lo:e], glp), f"env path: group ending at {e} (slot {s})"
        lo = e


@pytest.mark.timeout(300)
@pytest.mark.parametrize("n", [1000, 8192])
def test_one_group_is_the_pair_launch(eng, n):
    learner, other = _kernel(eng, 1), _kernel(eng, 2)
    pool = eng.OpponentPool(1)
    pool.add(other)
    x = torch.from_numpy(np.random.default_rng(n).normal(0, 1.5, (n, 18)).astype(np.float32)).cuda()
    kw = dict(obs=x, seed=99, step=4, other_step=5, row_offset=256)
    got = learner.sample_vs_pool(pool, [0], [n], tc=True, **kw)
    want = learner.sample_pair(other, tc=True, **kw)
    for g, w in zip(got, want):
        assert torch.equal(g, w)


def _args(B, mb, K=1):
    return types.SimpleNamespace(policy_dist="Gaussian", max_action=1.6, batch_size=B, mini_batch_size=mb, max_train_steps=int(3e6),
                                 lr_a=3e-3, lr_c=3e-3, gamma=0.99, lamda=0.95, epsilon=0.2, K_epochs=K, entropy_coef=0.01,
                                 set_adam_eps=True, use_grad_clip=True, use_lr_decay=False, use_adv_norm=True, state_dim=18,
                                 action_dim=3, hidden_width=256, use_tanh=1, use_orthogonal_init=True, chkpt_dir="/tmp")


def _agents(n, T, mb=512):
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    torch.manual_seed(0)
    a, b = P.PPO_continuous(_args(n * T, mb), "pursuer"), P.PPO_continuous(_args(n * T, mb), "evader")
    with torch.no_grad():                      # make the policy means matter
        for m in (a, b):
            m.actor.mean_layer.weight.mul_(30.0)
    a._dirty = b._dirty = True
    return a, b


def _box(dp=50000.0, dv=3.0):
    c = np.array(RESET_P + (0.0, 0.0, 0.0) + RESET_E + (0.0, 0.0, 0.0))
    d = np.array([dp] * 3 + [dv] * 3 + [dp] * 3 + [dv] * 3)
    return c - d, c + d


def _env(eng, n, row_offset=0):
    return eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=12, start_box=_box(), start_seed=21,
                        row_offset=row_offset)


@pytest.mark.timeout(300)
def test_snapshots_are_frozen(eng):
    from ppo_rl_satellite_b200 import rollout
    n, T, mb = 1024, 8, 512
    agent, opp = _agents(n, T, mb)
    tr = rollout.VectorTrainer(_env(eng, n), agent, opp, T, seed=3)
    tr.collect()                                 # syncs the kernels
    pool = eng.OpponentPool(2)
    pool.add(agent.actor_kernel)
    pool.add(opp.actor_kernel)
    x = torch.from_numpy(np.random.default_rng(0).normal(0, 1.5, (n, 18)).astype(np.float32)).cuda()
    kw = dict(obs=x, seed=1, step=2, other_step=3)
    before = [t.clone() for t in agent.actor_kernel.sample_vs_pool(pool, [0, 1], [512, n], tc=True, **kw)]
    tr.update(mb)                                # one fused PPO optimiser step on the learner
    after = agent.actor_kernel.sample_vs_pool(pool, [0, 1], [512, n], tc=True, **kw)
    assert torch.equal(after[2], before[2]) and torch.equal(after[3], before[3])     # the snapshots' rows
    assert not torch.equal(after[0], before[0])                                       # the learner's rows


_BUFS = ("obs", "act", "logp", "opp_act", "opp_logp", "rew64", "done", "ret_std")


@pytest.mark.timeout(300)
def test_pool_of_copies_changes_nothing(eng):
    from ppo_rl_satellite_b200 import rollout
    n, T = 8192, 8
    runs = []
    for use_pool in (False, True):
        agent, opp = _agents(n, T)
        pool = None
        if use_pool:
            opp.sync_kernels()
            pool = eng.OpponentPool(4)
            for _ in range(4):
                pool.add(opp.actor_kernel)
        tr = rollout.VectorTrainer(_env(eng, n), agent, opp, T, seed=5, opponent_pool=pool)
        tr.collect()
        runs.append(tr)
    for k in _BUFS:
        assert torch.equal(getattr(runs[0].buf, k), getattr(runs[1].buf, k)), k
    st = runs[1].opponent_stats
    assert [s["rows"] for s in st] == [2048] * 4 and sorted(s["snapshot_id"] for s in st) == [0, 1, 2, 3]


@pytest.mark.timeout(300)
def test_shards_equal_the_union(eng):
    from ppo_rl_satellite_b200 import rollout
    N, T, world = 8192, 6, 2
    snaps = [_kernel(eng, 200 + k) for k in range(4)]

    def pool():
        p = eng.OpponentPool(4)
        for k in snaps:
            p.add(k)
        return p

    def trainer(n, rank, w):
        agent, opp = _agents(n, T)
        return rollout.VectorTrainer(_env(eng, n, row_offset=rank * n), agent, opp, T, rank=rank, world=w, seed=7,
                                     use_state_norm=False, use_reward_scaling=False, opponent_pool=pool())

    union = trainer(N, 0, 1)
    shards = [trainer(N // world, r, world) for r in range(world)]
    for it in range(2):                          # two collects: two permutations
        union.collect()
        for s in shards:
            s.collect()
        for k in ("act", "logp", "opp_act", "opp_logp", "rew64", "done"):
            got = torch.cat([getattr(s.buf, k) for s in shards], dim=1)
            assert torch.equal(got, getattr(union.buf, k)), (it, k)
        ids = [(g["snapshot_id"], g["rows"]) for s in shards for g in s.opponent_stats]
        assert sum(r for _, r in ids) == N and {i for i, _ in ids} == {g["snapshot_id"] for g in union.opponent_stats}


@pytest.mark.timeout(600)
def test_selfplay_with_pools_and_resume(eng):
    from ppo_rl_satellite_b200 import rollout
    n, T, mb = 512, 4, 512
    sp = rollout.SelfPlay(_env(eng, n), *_agents(n, T, mb), T, mb, seed=11, opponent_pool=4)
    assert [len(sp.pools[0]), len(sp.pools[1])] == [1, 1]
    log = sp.run(2, 1)
    assert [len(sp.pools[0]), len(sp.pools[1])] == [3, 3]
    assert sp.pools[0].ids == [0, 1, 2] and sp.pools[1].ids == [0, 1, 2]
    sizes = {0: 1, 1: 2}                          # opponent pool size seen by each phase of round 1
    for i, rec in enumerate(log):
        opps = rec["opponents"]
        assert sum(o["rows"] for o in opps) == n
        assert all(set(o) == {"snapshot_id", "rows", "mean_reward", "episodes_finished"} for o in opps)
        want = sizes[rec["flag"]] + (i // 2)                      # each round adds one snapshot to each pool
        assert len(opps) == want, (i, rec["flag"], len(opps))
    sp.pools[0].add(sp.trainers[0].agent.actor_kernel)            # 4 snapshots; a fifth evicts the oldest
    sp.pools[0].add(sp.trainers[0].agent.actor_kernel)
    assert sp.pools[0].ids == [1, 2, 3, 4]

    # checkpoint: a fresh trainer resumes to the same next collect()
    sp.env.reset(flag=0)
    tr = sp.trainers[0]
    tr.learner_is_pursuer = True
    sd = copy.deepcopy(tr.state_dict())
    assert sd["collects"] == 2 and sd["opponent_pool"]["ids"] == [0, 1, 2]
    tr.collect()
    a2, b2 = _agents(n, T, mb)
    fresh = rollout.VectorTrainer(_env(eng, n), a2, b2, T, seed=11, opponent_pool=eng.OpponentPool(4)).load_state_dict(sd)
    assert fresh.opponent_pool.ids == [0, 1, 2]
    fresh.collect()
    for k in _BUFS:
        assert torch.equal(getattr(tr.buf, k), getattr(fresh.buf, k)), k
    assert tr.opponent_stats == fresh.opponent_stats


@pytest.mark.timeout(300)
def test_argument_checks(eng):
    L = eng.L
    lib = L.load()
    n = 1024
    learner, relu = _kernel(eng, 1), _kernel(eng, 2, use_tanh=False)
    pool = _pool(eng, 3)
    x = torch.zeros((n, 18), dtype=torch.float32, device="cuda")
    a, lp, oa, olp = _outs(n, 4)

    def call(groups, ends, w=learner.w, n_=n, act_b=oa):
        arr = (L.SatActorPoolGroup * max(1, len(groups)))()
        for k, (g, e) in enumerate(zip(groups, ends)):
            arr[k] = g
            arr[k].row_end = e
        return lib.sat_actor_sample_pool_tc(C.byref(w), learner._image().data_ptr(), arr, len(groups), L.ptr(x), None, None,
                                            n_, 0, 1, 2, 3, L.ptr(a), L.ptr(lp), None, L.ptr(act_b), L.ptr(olp),
                                            L.stream_ptr())

    g = [pool.group(k) for k in range(3)]
    assert call(g, [256, 512, n]) == 0
    torch.cuda.synchronize()
    # SAT_ERR_NULL
    assert call(g, [256, 512, n], w=L.SatActorWeights()) == -1
    assert call(g, [256, 512, n], act_b=None) == -1
    bad = L.SatActorPoolGroup.from_buffer_copy(g[1]); bad.packed = None
    assert call([g[0], bad, g[2]], [256, 512, n]) == -1
    assert lib.sat_actor_sample_pool_tc(C.byref(learner.w), learner._image().data_ptr(), None, 1, L.ptr(x), None, None, n,
                                        0, 1, 2, 3, L.ptr(a), L.ptr(lp), None, L.ptr(oa), L.ptr(olp), L.stream_ptr()) == -1
    snap = L.SatActorPoolGroup()
    tab = torch.empty(L.ACTOR_TC_TABLE_FLOATS, dtype=torch.float32, device="cuda")
    assert lib.sat_actor_tc_snapshot(C.byref(learner.w), None, tab.data_ptr(), C.byref(snap), L.stream_ptr()) == -1
    # SAT_ERR_SIZE
    assert call([], []) == -2
    assert call([g[0]] * 17, [128 * (k + 1) for k in range(16)] + [n]) == -2
    assert call(g, [512, 256, n]) == -2                              # not increasing
    assert call(g, [512, 512, n]) == -2                              # empty group
    assert call(g, [200, 512, n]) == -2                              # interior bound off the 128-row tile
    assert call(g, [256, 512, n - 1]) == -2                          # last bound != n
    mis = L.SatActorPoolGroup.from_buffer_copy(g[1]); mis.tc_image = g[1].tc_image + 4
    assert call([g[0], mis, g[2]], [256, 512, n]) == -2              # misaligned image
    assert lib.sat_actor_tc_snapshot(C.byref(learner.w), learner._image().data_ptr() + 4, tab.data_ptr(), C.byref(snap),
                                     L.stream_ptr()) == -2
    # SAT_ERR_MODE: a ReLU snapshot for a tanh learner
    rpool = _pool(eng, 1, use_tanh=False)
    assert call([g[0], rpool.group(0), g[2]], [256, 512, n]) == -3
    torch.cuda.synchronize()

    # the same codes through sample_vs_pool
    kw = dict(obs=x, tc=True)
    nulled = copy.copy(learner); nulled.w = L.SatActorWeights()
    with pytest.raises(L.SatError, match=r"code -1\)"):
        nulled.sample_vs_pool(pool, [0, 1, 2], [256, 512, n], **kw)
    for ends in ([512, 256, n], [200, 512, n], [256, 512, n - 1]):
        with pytest.raises(L.SatError, match=r"code -2\)"):
            learner.sample_vs_pool(pool, [0, 1, 2], ends, **kw)
    with pytest.raises(L.SatError, match=r"code -3\)"):
        relu.sample_vs_pool(pool, [0], [n], **kw)
    with pytest.raises(L.SatError):
        pool.add(relu)                                               # a pool holds one activation
    with pytest.raises(L.SatError):                                  # FFMA2 path: the same checks in Python
        learner.sample_vs_pool(pool, [0, 1, 2], [200, 512, n], obs=x, tc=False)
