"""Per-env start states of EnvBatch (start_box): the device draw against a numpy restatement of its exact mapping, the
in-kernel auto-reset to the starts against the oracle (cw and rk4 mode), and the batch / trainer semantics built on them.
All tests but the Philox known-answer test need a GPU."""
import copy
import ctypes as C
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

gpu = pytest.mark.gpu

MASK32 = np.uint64(0xFFFFFFFF)
RESET_P, RESET_E = (200000.0, 0.0, 0.0), (18000.0, 0.0, 0.0)


# ------------------------------------------------------------------------------------------------ host restatements
def philox4x32_10(c, k0, k1):
    """Philox4x32-10 over numpy uint64 arrays holding 32-bit words (the round structure of sat::philox4x32_10)"""
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) & MASK32 for x in c)
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & MASK32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & MASK32
        k0 = (k0 + np.uint64(0x9E3779B9)) & MASK32
        k1 = (k1 + np.uint64(0xBB67AE85)) & MASK32
    return c0, c1, c2, c3


def draw_starts_ref(n, lo, hi, seed, draw, row_offset):
    """[12, n] starts sat_env_draw_starts writes for envs 0..n-1 (every env drawn)"""
    g = np.arange(n, dtype=np.uint64) + np.uint64(row_offset)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) ^ 0x53434E31
    out = np.empty((12, n))
    for j in range(6):
        c = philox4x32_10((g & MASK32, g >> np.uint64(32), np.full(n, draw, dtype=np.uint64), np.full(n, j, dtype=np.uint64)),
                          k0, k1)
        for h in range(2):
            col = 2 * j + h
            bits = ((c[2 * h] << np.uint64(32)) | c[2 * h + 1]) >> np.uint64(11)
            u = bits.astype(np.float64) * 2.0 ** -53
            if lo[col] < hi[col]:
                out[col] = np.minimum(lo[col] + (hi[col] - lo[col]) * u, hi[col])
            else:
                out[col] = lo[col]
    return out


def obs_of(S):
    """observation [n, 18] of kinematics S [12, n] (environment.py:76-77)"""
    P, Pv, E, Ev = S[0:3].T, S[3:6].T, S[6:9].T, S[9:12].T
    return np.concatenate([P - E, Pv - Ev, P, Pv, E, Ev], axis=1)


def box(dp=50000.0, dv=3.0):
    """+-dp around the reference's reset positions, +-dv on every velocity component"""
    c = np.array(RESET_P + (0.0, 0.0, 0.0) + RESET_E + (0.0, 0.0, 0.0))
    d = np.array([dp] * 3 + [dv] * 3 + [dp] * 3 + [dv] * 3)
    return c - d, c + d


def test_philox_known_answer_vectors():
    """Random123's published known-answer vectors for philox4x32_10"""
    cases = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
             ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
              (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in cases:
        got = philox4x32_10([np.array([x], dtype=np.uint64) for x in ctr], *key)
        assert tuple(int(x[0]) for x in got) == want


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def eng():
    from ppo_rl_satellite_b200 import engine
    return engine


@pytest.fixture(scope="module")
def L():
    from ppo_rl_satellite_b200 import _lib
    return _lib


def _cw_kw(golden, **kw):
    return dict(mode="cw", stm=golden("env_golden.npz")["stm100_columns"], **kw)


def _actions(rng, n, integer=False):
    if integer:
        return [rng.integers(-1, 2, (n, 3)).astype(np.float32) for _ in range(2)]
    return [rng.uniform(-2, 2, (n, 3)).astype(np.float32) for _ in range(2)]


def _orc_reset_rows(orc, rows, S):
    """the starts-mode reset on oracle envs: kinematics from S [12, n], int_state 0, count 0"""
    for i in rows:
        e = orc.envs[int(i)]
        for k in range(3):
            e.P[k], e.Pv[k], e.E[k], e.Ev[k] = S[k, i], S[3 + k, i], S[6 + k, i], S[9 + k, i]
        e.int_state = 0
        orc.counts[int(i)] = 0


@gpu
def test_draw_matches_host_restatement_bit_for_bit(eng, L):
    n = 65536 + 37
    lo, hi = box()
    lo[4] = hi[4] = 1.25                     # fixed columns: exactly lo
    lo[8] = hi[8] = -7.0e3
    env = eng.EnvBatch(n, start_box=(lo, hi))
    lib = L.load()
    rng = np.random.default_rng(21)
    blo, bhi = (C.c_double * 12)(*lo), (C.c_double * 12)(*hi)
    half = torch.from_numpy((rng.random(n) < 0.5).astype(np.uint8)).cuda()
    masks = {"null": None, "all": torch.ones(n, dtype=torch.uint8, device="cuda"), "half": half,
             "none": torch.zeros(n, dtype=torch.uint8, device="cuda")}
    row_offset = (1 << 33) + 12345                     # non-zero high word of the global id
    for seed in (0, 0xDEADBEEF12345678):
        for draw in (0, 0xFFFFFFFE):
            want = draw_starts_ref(n, lo, hi, seed, draw, row_offset)
            for name, m in masks.items():
                env.state.copy_(torch.from_numpy(rng.normal(0, 1e5, env.state.shape)))
                env.istate.copy_(torch.from_numpy(rng.integers(-9, 9, env.istate.shape).astype(np.int32)))
                before, ibefore = env.state.cpu().numpy(), env.istate.cpu().clone()
                L.check(lib.sat_env_draw_starts(C.byref(env.st), L.ptr(m), blo, bhi, seed, draw, row_offset, L.stream_ptr()))
                got = env.state.cpu().numpy()
                sel = np.ones(n, bool) if m is None else m.cpu().numpy().astype(bool)
                assert np.array_equal(got[16:, sel].view(np.int64), want[:, sel].view(np.int64)), (seed, draw, name)
                assert np.array_equal(got[16:, ~sel].view(np.int64), before[16:, ~sel].view(np.int64))
                assert np.array_equal(got[:16].view(np.int64), before[:16].view(np.int64))
                assert torch.equal(env.istate.cpu(), ibefore)
                if sel.any():
                    assert np.all(got[16 + 4, sel] == 1.25) and np.all(got[16 + 8, sel] == -7.0e3)
                    assert np.all((got[16:, sel] >= lo[:, None]) & (got[16:, sel] <= hi[:, None]))
    # argument errors
    st = C.byref(env.st)
    assert lib.sat_env_draw_starts(st, None, None, bhi, 0, 0, 0, None) == -1
    assert lib.sat_env_draw_starts(st, None, blo, None, 0, 0, 0, None) == -1
    assert lib.sat_env_draw_starts(st, None, blo, bhi, 0, 0, -1, None) == -2
    for bad in (lambda a, b: a.__setitem__(3, b[3] + 1.0), lambda a, b: a.__setitem__(0, float("nan")),
                lambda a, b: a.__setitem__(5, float("-inf"))):
        a = (C.c_double * 12)(*lo)
        bad(a, hi)
        assert lib.sat_env_draw_starts(st, None, a, bhi, 0, 0, 0, None) == -2
    h2 = (C.c_double * 12)(*hi); h2[7] = float("inf")
    assert lib.sat_env_draw_starts(st, None, blo, h2, 0, 0, 0, None) == -2
    empty = L.SatEnvState(env.st.state, env.st.istate, 0, env.st.ld)
    assert lib.sat_env_draw_starts(C.byref(empty), None, blo, bhi, 0, 0, 0, None) == -2
    assert lib.sat_env_reset_starts(C.byref(empty), None, None) == -2
    nul = L.SatEnvState(None, env.st.istate, n, env.st.ld)
    assert lib.sat_env_reset_starts(C.byref(nul), None, None) == -1
    with pytest.raises(L.SatError):
        eng.EnvBatch(4, start_box=(lo[:11], hi[:11]))
    with pytest.raises(L.SatError):
        eng.EnvBatch(4, start_box=(hi, lo))


@gpu
@pytest.mark.parametrize("flag", [0, 1])
def test_cw_starts_mode_bit_identical_to_oracle(golden, oracle, eng, flag):
    """2048 envs x 160 steps: the auto-reset to each env's start, emulated on the oracle from a snapshot of the starts taken
    before every step. Observations (next and pre-reset), rewards and dones bit for bit, no danger-zone flips."""
    n, T = 2048, 160
    kw = dict(d_capture=181200.0, max_episode_steps=40, flag=flag)
    env = eng.EnvBatch(n, start_box=box(), start_seed=7 + flag, **_cw_kw(golden, **kw))
    orc = oracle.BatchEnv(n, nthreads=8, M=golden("env_golden.npz")["stm100_columns"], **kw)
    S0 = env.state[:12].cpu().numpy()
    orc.set_state(S0[0:3].T, S0[3:6].T, S0[6:9].T, S0[9:12].T)
    assert len(np.unique(S0[0])) > n // 2
    rng = np.random.default_rng(200 + flag)
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    term = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    n_done = n_dz = 0
    for t in range(T):
        starts = env.starts.cpu().numpy()
        pa, ea = _actions(rng, n)
        r, d = env.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f64=obs, term_obs_f64=term)
        o_obs, o_r, o_d = orc.step(pa.astype(np.float64), ea.astype(np.float64), auto_reset=False)
        dn = o_d.astype(bool)
        assert np.array_equal(d.cpu().numpy(), o_d), t
        assert np.array_equal(r.cpu().numpy(), o_r), t
        assert np.array_equal(term.cpu().numpy(), o_obs), t
        _orc_reset_rows(orc, np.flatnonzero(dn), starts)
        o_obs[dn] = obs_of(starts)[dn]
        assert np.array_equal(obs.cpu().numpy(), o_obs), t
        n_dz += int((env.dangerous_zone.cpu().numpy() != orc.aux()[3]).sum())
        n_done += int(dn.sum())
        if dn.any():                             # the finished envs' next starts were redrawn, the others kept
            now = env.starts.cpu().numpy()
            assert np.array_equal(now[:, ~dn], starts[:, ~dn])
            assert np.all(now[0, dn] != starts[0, dn])
    assert n_done > 1000
    assert n_dz == 0
    assert int(env.err.sum()) == 0
    assert np.array_equal(env.state[:12].cpu().numpy(), orc.state().T)


@gpu
def test_degenerate_box_reproduces_the_default_batch(golden, eng):
    """lo == hi == the reset literals and integer actions (the int64 truncation is then the identity): starts mode equals
    the default batch in everything but int_state"""
    n, T = 1024, 120
    c = np.array(RESET_P + (0.0,) * 3 + RESET_E + (0.0,) * 3)
    kw = _cw_kw(golden, d_capture=181200.0, max_episode_steps=30)
    a = eng.EnvBatch(n, **kw)
    b = eng.EnvBatch(n, start_box=(c, c), **kw)
    assert np.array_equal(b.starts.cpu().numpy(), np.repeat(c[:, None], n, axis=1))
    rng = np.random.default_rng(4)
    oa, ob = (torch.empty((n, 18), dtype=torch.float64, device="cuda") for _ in range(2))
    dones = 0
    for t in range(T):
        pa, ea = (torch.from_numpy(x).cuda() for x in _actions(rng, n, integer=True))
        ra, da = a.step(pa, ea, obs_f64=oa)
        rb, db = b.step(pa, ea, obs_f64=ob)
        assert torch.equal(da, db) and torch.equal(ra, rb) and torch.equal(oa, ob), t
        assert torch.equal(a.state, b.state[:16]), t
        for col in (0, 1, 3):                                  # dangerous_zone, count, err
            assert torch.equal(a.istate[col], b.istate[col]), t
        dones += int(da.sum())
    assert dones > n


@gpu
def test_rk4_starts_mode_vs_oracle_and_input_selected_host_forms(oracle, eng):
    """rk4 mode: the device step against the oracle's step_rk4 with the auto-reset to the starts emulated (tolerances of
    test_env_rk4_mode_vs_oracle); then every host-buffer form equals the device-resident starts-mode step"""
    n, T, S = 512, 16, 20
    kw = dict(d_capture=20000.0, max_episode_steps=5)
    env = eng.EnvBatch(n, mode="rk4", substeps=S, h=1.0, start_box=box(), start_seed=3, **kw)
    orc = oracle.BatchEnv(n, nthreads=8, **kw)
    S0 = env.state[:12].cpu().numpy()
    orc.set_state(S0[0:3].T, S0[3:6].T, S0[6:9].T, S0[9:12].T)
    rng = np.random.default_rng(13)
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    R = np.array([27098000.0, 32306000.0, 0.0]); V = np.array([-2350.0, 1970.0, 0.0])
    diverged = np.zeros(n, dtype=bool)
    resets = 0
    for t in range(T):
        starts = env.starts.cpu().numpy()
        pa, ea = _actions(rng, n)
        r, d = env.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f64=obs)
        o_obs, o_r, o_d = orc.step_rk4(pa.astype(np.float64), ea.astype(np.float64), h=1.0, substeps=S, auto_reset=False)
        dn = o_d.astype(bool)
        _orc_reset_rows(orc, np.flatnonzero(dn), starts)
        o_obs[dn] = obs_of(starts)[dn]
        dz_same = env.dangerous_zone.cpu().numpy() == orc.aux()[3]
        ok = ~diverged
        assert np.array_equal(d.cpu().numpy()[ok], o_d[ok])
        got = obs.cpu().numpy()
        assert np.array_equal(got[ok & dn], o_obs[ok & dn])            # post-reset observations are the starts exactly
        for lo in (6, 12):
            dr = np.linalg.norm(got[ok, lo:lo + 3] - o_obs[ok, lo:lo + 3], axis=1) / np.linalg.norm(o_obs[ok, lo:lo + 3] + R, axis=1)
            dv = np.linalg.norm(got[ok, lo + 3:lo + 6] - o_obs[ok, lo + 3:lo + 6], axis=1) / np.linalg.norm(o_obs[ok, lo + 3:lo + 6] + V, axis=1)
            assert dr.max() < 1e-9 and dv.max() < 1e-9, (t, dr.max(), dv.max())
        both = ok & dz_same
        np.testing.assert_allclose(r.cpu().numpy()[both], o_r[both], rtol=0, atol=1e-6)
        diverged |= ~dz_same
        resets += int((dn & ok).sum())
    assert diverged.mean() < 0.02, diverged.mean()
    assert resets > n

    from test_gpu_parity import step_host_call
    n = 1500
    hkw = dict(mode="rk4", substeps=5, h=1.0, d_capture=150000.0, max_episode_steps=6, start_box=box(60000.0, 3.0), start_seed=9)
    for form in ("overlapped", "zero-copy", "staged"):
        a, b = eng.EnvBatch(n, **hkw), eng.EnvBatch(n, **hkw)
        obs_d = torch.empty((n, 18), dtype=torch.float32, device="cuda")
        dones = 0
        for t in range(9):
            pa, ea = _actions(rng, n)
            r, d = a.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f32=obs_d)
            if form == "overlapped":
                o, rh, dh = b.step_host(pa, ea)
            else:
                o, rh, dh = step_host_call(b, pa, ea, pinned=form == "zero-copy")
            assert np.array_equal(dh, d.cpu().numpy()) and np.array_equal(rh, r.cpu().numpy()), (form, t)
            assert np.array_equal(o, obs_d.cpu().numpy()), (form, t)
            dones += int(dh.sum())
        assert dones > n
        assert torch.equal(a.state, b.state) and torch.equal(a.istate, b.istate) and a.start_draws == b.start_draws


@gpu
def test_running_statistics_see_the_post_reset_observations(golden, oracle, eng):
    n = 300
    env = eng.EnvBatch(n, start_box=box(), start_seed=5, gamma=0.99, **_cw_kw(golden, d_capture=20000.0, max_episode_steps=9))
    obs_stats, ret_stats = eng.RunningStats(18), eng.RunningStats(1)
    std_out = torch.zeros(1, dtype=torch.float64, device="cuda")
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    rng = np.random.default_rng(8)
    cnt, mean, S = 0, np.zeros(18), np.zeros(18)
    rc, rmean, rS = 0, np.zeros(1), np.zeros(1)
    R = np.zeros(n)
    dones = 0
    for t in range(25):
        starts = env.starts.cpu().numpy()
        pa, ea = (torch.from_numpy(x).cuda() for x in _actions(rng, n))
        r, d = env.step(pa, ea, obs_f64=obs, obs_stats=obs_stats, ret_stats=ret_stats, ret_std_out=std_out)
        x = obs.cpu().numpy()
        dn = d.cpu().numpy().astype(bool)
        assert np.array_equal(x[dn], obs_of(starts)[dn])
        dones += int(dn.sum())
        cnt, mean, S = oracle.chan_merge(cnt, mean, S, x)
        R = 0.99 * R + r.cpu().numpy()
        rc, rmean, rS = oracle.chan_merge(rc, rmean, rS, R[:, None])
        R[dn] = 0.0
        np.testing.assert_allclose(obs_stats.mean.cpu().numpy(), mean, rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(obs_stats.S.cpu().numpy(), S, rtol=1e-10, atol=1e-5)
        np.testing.assert_allclose(ret_stats.S.cpu().numpy(), rS, rtol=1e-10, atol=1e-8)
        np.testing.assert_allclose(float(std_out[0]), np.sqrt(rS[0] / rc), rtol=1e-12)
    assert dones > n
    assert obs_stats.n == 25 * n and ret_stats.n == 25 * n


@gpu
def test_shards_draw_and_roll_out_like_one_batch(golden, eng):
    n, T = 4096, 50
    kw = dict(start_box=box(), start_seed=0xABCDEF0123, **_cw_kw(golden, d_capture=181200.0, max_episode_steps=12))
    full = eng.EnvBatch(n, **kw)
    parts = [eng.EnvBatch(n // 2, row_offset=k * (n // 2), **kw) for k in range(2)]
    cat = lambda f: torch.cat([f(p) for p in parts], dim=-1)
    assert torch.equal(full.state, cat(lambda p: p.state))
    rng = np.random.default_rng(17)
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    po = [torch.empty((n // 2, 18), dtype=torch.float64, device="cuda") for _ in parts]
    dones = 0
    for t in range(T):
        pa, ea = (torch.from_numpy(x).cuda() for x in _actions(rng, n))
        r, d = full.step(pa, ea, obs_f64=obs)
        outs = [p.step(pa[k * n // 2:(k + 1) * n // 2].contiguous(), ea[k * n // 2:(k + 1) * n // 2].contiguous(), obs_f64=po[k])
                for k, p in enumerate(parts)]
        assert torch.equal(r, torch.cat([o[0] for o in outs])) and torch.equal(d, torch.cat([o[1] for o in outs])), t
        assert torch.equal(obs, torch.cat(po)), t
        dones += int(d.sum())
    assert torch.equal(full.state, cat(lambda p: p.state)) and torch.equal(full.istate, cat(lambda p: p.istate))
    assert dones > n


@gpu
def test_reset_mask_semantics(golden, eng):
    n = 5000
    lo, hi = box()
    env = eng.EnvBatch(n, start_box=(lo, hi), start_seed=77, **_cw_kw(golden, d_capture=20000.0, max_episode_steps=1000))
    assert env.start_draws == 2
    rng = np.random.default_rng(2)
    for t in range(6):                                       # fuel, dis, dangerous_zone and the return move away from reset values
        env.step(*(torch.from_numpy(x).cuda() for x in _actions(rng, n)))
    s0, i0 = env.state.cpu().numpy(), env.istate.cpu().numpy()
    m = (rng.random(n) < 0.5).astype(np.uint8)
    sel = m.astype(bool)
    draw = env.start_draws
    env.reset(torch.from_numpy(m).cuda())
    assert env.start_draws == draw + 1
    s1, i1 = env.state.cpu().numpy(), env.istate.cpu().numpy()
    assert np.array_equal(s1[:12, sel], s0[16:, sel])                        # kinematics = the previous starts
    assert np.all(i1[1, sel] == 0) and np.all(i1[2, sel] == 0)               # count, int_state
    assert np.array_equal(s1[12:16], s0[12:16])                              # fuel, dis, return persist
    assert np.array_equal(i1[0], i0[0]) and np.array_equal(i1[3], i0[3])     # dangerous_zone, err
    assert np.array_equal(s1[:12, ~sel], s0[:12, ~sel]) and np.array_equal(i1[:, ~sel], i0[:, ~sel])
    assert np.array_equal(s1[16:, ~sel], s0[16:, ~sel])                      # unmasked starts untouched
    want = draw_starts_ref(n, lo, hi, 77, draw, 0)
    assert np.array_equal(s1[16:, sel], want[:, sel])                        # masked starts redrawn with the next index
    assert np.all(s1[16, sel] != s0[16, sel])


def _args(K=2, mb=512, B=2048):
    return types.SimpleNamespace(policy_dist="Gaussian", max_action=1.6, batch_size=B, mini_batch_size=mb, max_train_steps=int(3e6),
                                 lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1, K_epochs=K, entropy_coef=0.01,
                                 set_adam_eps=True, use_grad_clip=True, use_lr_decay=True, use_adv_norm=True, state_dim=18,
                                 action_dim=3, hidden_width=256, use_tanh=1, use_orthogonal_init=True, chkpt_dir="/tmp")


@gpu
def test_vector_trainer_on_starts_mode(eng):
    from ppo_rl_satellite_b200 import rollout
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    n, T, mb = 256, 8, 512

    def make(norm=True):
        torch.manual_seed(0)
        env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=3, start_box=box(), start_seed=11)
        agent, opp = P.PPO_continuous(_args(mb=mb, B=n * T), "pursuer"), P.PPO_continuous(_args(mb=mb, B=n * T), "evader")
        return rollout.VectorTrainer(env, agent, opp, T, use_state_norm=norm)

    # raw observations: every env starts elsewhere, and each new episode starts elsewhere than the last
    raw = make(norm=False)
    raw.collect()
    o, dn = raw.buf.obs.cpu().numpy(), raw.buf.done.cpu().numpy().astype(bool)
    assert len(np.unique(o[0, :, 6])) > n // 2
    first = np.argmax(dn, axis=0)
    assert dn.any(axis=0).all()
    rows = np.arange(n)
    assert np.all(np.any(o[first + 1, rows] != o[0, rows], axis=1))

    a = make()
    a.collect(); torch.manual_seed(5); a.update(mb, total_steps=1000)
    sd = copy.deepcopy(a.state_dict())
    assert sd["env"]["start_box"] is not None and sd["env"]["start_draws"] == a.env.start_draws
    a.collect(); torch.manual_seed(6); a.update(mb, total_steps=2000)
    b = make().load_state_dict(sd)
    b.collect(); torch.manual_seed(6); b.update(mb, total_steps=2000)
    for pa, pb in zip(list(a.agent.actor.parameters()) + list(a.agent.critic.parameters()),
                      list(b.agent.actor.parameters()) + list(b.agent.critic.parameters())):
        assert torch.equal(pa, pb)
    assert torch.equal(a.buf.act, b.buf.act) and torch.equal(a.buf.rew64, b.buf.rew64) and torch.equal(a.buf.obs, b.buf.obs)
    assert torch.equal(a.env.state, b.env.state) and torch.equal(a.env.istate, b.env.istate)
    assert a.env.start_draws == b.env.start_draws
    with pytest.raises(eng.L.SatError):                     # a default-mode batch refuses a starts-mode checkpoint
        eng.EnvBatch(n, mode="cw").load_state_dict(sd["env"])

    # SelfPlay's phase reset goes through the starts: every env at its start, one draw for the reset and one per step
    sp = rollout.SelfPlay(make().env, *(P.PPO_continuous(_args(mb=mb, B=n * 4), r) for r in ("pursuer", "evader")), 4, mb)
    env = sp.env
    starts, draws = env.starts.cpu().numpy(), env.start_draws
    env.reset(flag=1)
    assert np.array_equal(env.state[:12].cpu().numpy(), starts) and env.start_draws == draws + 1
    assert int(env.istate[2].sum()) == 0 and env.params.flag == 1
    sp.run_phase(0, 1)
    assert env.start_draws == draws + 2 + 4
