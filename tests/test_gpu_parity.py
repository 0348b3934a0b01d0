"""GPU parity tests: the CUDA path (through the C ABI) against the reference-generated golden
fixtures and against the CPU oracle on seeded inputs. Run on the B200 box: pytest -m gpu."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def eng():
    from ppo_rl_satellite_b200 import engine
    return engine


def rel_err_rv(x, y):
    dr = np.linalg.norm(x[:3] - y[:3], axis=0) / np.linalg.norm(y[:3], axis=0)
    dv = np.linalg.norm(x[3:] - y[3:], axis=0) / np.linalg.norm(y[3:], axis=0)
    return max(dr.max(), dv.max())


def soa(x_np, eng):
    view, _buf = eng.alloc_soa(6, x_np.shape[1], torch.float64, "cuda")
    view.copy_(torch.from_numpy(np.ascontiguousarray(x_np)))
    return view


# ============================================================================ K1: RK4 propagator
@pytest.mark.parametrize("tag,j2", [("j2off", 0.0), ("j2on", 0.00108263)])
def test_rk4_config2_vs_reference_golden(golden, eng, tag, j2):
    """BASELINE config 2: 4096 LEO/GEO orbits x 1000 steps of 1 s; bar 1e-9 relative (north star)."""
    g = golden("rk4_golden.npz")
    x = soa(g["x0"], eng)
    eng.rk4_propagate(x, 1.0, 1000, j2=j2)                   # one launch, 1000 substeps in registers
    err = rel_err_rv(x.cpu().numpy(), g[f"x1000_{tag}"])
    assert err < 1e-9, err
    assert err < 1e-11, f"expected ~1e-13 headroom, got {err}"
    y = soa(g["x0"], eng)
    for _ in range(1000):                                    # 1000 launches of one step (the script's loop shape)
        eng.rk4_propagate(y, 1.0, 1, j2=j2)
    assert rel_err_rv(y.cpu().numpy(), g[f"x1000_{tag}"]) < 1e-9
    assert torch.equal(x, y)                                 # substep batching does not change a bit


def test_rk4_script_initial_condition(golden, eng):
    g = golden("rk4_golden.npz")
    x = soa(g["script_ic"].reshape(6, 1), eng)
    eng.rk4_propagate(x, 1.0, 86400)
    assert rel_err_rv(x.cpu().numpy(), g["script_86400"].reshape(6, 1)) < 1e-9


@pytest.mark.parametrize("n", [1, 33, 151552 + 7])
def test_rk4_vs_oracle_ragged_sizes(golden, oracle, eng, n):
    """edge sizes incl. the two-states-per-thread path with an odd tail; oracle = literal C restatement."""
    g = golden("rk4_golden.npz")
    reps = -(-n // 4096)
    x0 = np.tile(g["x0"], (1, reps))[:, :n].copy()
    x0 *= 1.0 + 1e-6 * np.random.default_rng(n).standard_normal(x0.shape)
    steps = 25
    x = soa(x0, eng)
    eng.rk4_propagate(x, 1.0, steps)
    ref = oracle.rk4_propagate(x0, 1.0, steps, nthreads=8)
    assert rel_err_rv(x.cpu().numpy(), ref) < 1e-12


def test_rk4_energy_and_momentum_conserved(golden, eng):
    g = golden("rk4_golden.npz")
    x0 = g["x0"]
    x = soa(x0, eng)
    eng.rk4_propagate(x, 1.0, 1000, j2=0.0)
    x1 = x.cpu().numpy()
    mu = 398600.0

    def energy(s):
        return 0.5 * (s[3:] ** 2).sum(0) - mu / np.linalg.norm(s[:3], axis=0)

    def hvec(s):
        return np.cross(s[:3].T, s[3:].T)
    assert np.max(np.abs(energy(x1) / energy(x0) - 1)) < 1e-10
    assert np.max(np.linalg.norm(hvec(x1) - hvec(x0), axis=1) / np.linalg.norm(hvec(x0), axis=1)) < 1e-12


def test_rk4_host_buffer_form(golden, eng):
    g = golden("rk4_golden.npz")
    prop = eng.Rk4HostPropagator(4096)
    out = prop(g["x0"], 1.0, 1000)
    assert rel_err_rv(out, g["x1000_j2on"]) < 1e-9


def test_rk4_argument_errors(eng):
    from ppo_rl_satellite_b200 import _lib as L
    lib = L.load()
    assert lib.sat_rk4_propagate(None, 4, 4, 1.0, 1, 1.0, 1.0, 0.0, None) == -1
    x = torch.zeros((6, 4), dtype=torch.float64, device="cuda")
    assert lib.sat_rk4_propagate(x.data_ptr(), 4, 3, 1.0, 1, 1.0, 1.0, 0.0, None) == -2   # ld < n
    assert lib.sat_rk4_propagate(x.data_ptr(), 0, 4, 1.0, 1, 1.0, 1.0, 0.0, None) == -2
    assert b"NULL" in lib.sat_strerror(-1)


# ============================================================================ K2: env step (cw = shipped env)
@pytest.mark.parametrize("scen", ["cfg1", "long", "capt", "flag1"])
def test_env_cw_bit_identical_to_reference_rollouts(golden, eng, scen):
    """N=1 env driven by the reference's recorded action stream: obs, reward, done, danger-zone count,
    fuel and distance must be IDENTICAL to the reference env (north star: rewards/dones identical)."""
    g = {**golden("env_golden.npz"), **golden("env_capt_golden.npz")}
    T = len(g[f"{scen}_reward"])
    env = eng.EnvBatch(1, mode="cw", flag=int(g[f"{scen}_flag"]), d_capture=float(g[f"{scen}_d_capture"]),
                       max_episode_steps=int(g[f"{scen}_max_episode_steps"]), auto_reset=True, stm=g["stm100_columns"])
    assert np.array_equal(env.observe().cpu().numpy()[0], g[f"{scen}_reset_obs"])
    pa = torch.from_numpy(g[f"{scen}_pa"]).cuda()
    ea = torch.from_numpy(g[f"{scen}_ea"]).cuda()
    term = torch.empty((T, 1, 18), dtype=torch.float64, device="cuda")
    rew = torch.empty((T, 1), dtype=torch.float64, device="cuda")
    done = torch.empty((T, 1), dtype=torch.uint8, device="cuda")
    aux = torch.empty((T, 4), dtype=torch.float64, device="cuda")
    for t in range(T):
        env.step(pa[t:t + 1], ea[t:t + 1], term_obs_f64=term[t], reward=rew[t], done=done[t])
        aux[t, 0] = env.dangerous_zone[0]; aux[t, 1] = env.fuel_c[0]; aux[t, 2] = env.fuel_t[0]; aux[t, 3] = env.dis[0]
    term, rew, done, aux = term.cpu().numpy()[:, 0], rew.cpu().numpy()[:, 0], done.cpu().numpy()[:, 0], aux.cpu().numpy()
    assert np.array_equal(done.astype(bool), g[f"{scen}_done"])
    assert np.array_equal(aux[:, 0].astype(np.int32), g[f"{scen}_dz"])
    assert np.array_equal(term, g[f"{scen}_obs"])
    assert np.array_equal(rew, g[f"{scen}_reward"])
    assert np.array_equal(aux[:, 1], g[f"{scen}_fuel_c"]) and np.array_equal(aux[:, 2], g[f"{scen}_fuel_t"])
    assert np.array_equal(aux[:, 3], g[f"{scen}_dis"])
    assert int(env.err[0]) == 0


def test_env_cw_explicit_episode_count_matches_reference_signature(golden, eng):
    """step(pa, ea, epsiode_count): the count argument of the reference overrides the internal counter."""
    g = golden("env_golden.npz")
    env = eng.EnvBatch(1, mode="cw", d_capture=20000.0, max_episode_steps=64, auto_reset=False, stm=g["stm100_columns"])
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    obs = torch.empty((1, 18), dtype=torch.float64, device="cuda")
    for t in range(70):
        cnt[0] = int(g["cfg1_count"][t])
        r, d = env.step(torch.from_numpy(g["cfg1_pa"][t:t + 1]).cuda(), torch.from_numpy(g["cfg1_ea"][t:t + 1]).cuda(),
                        count=cnt, obs_f64=obs)
        assert np.array_equal(obs.cpu().numpy()[0], g["cfg1_obs"][t])
        assert float(r[0]) == g["cfg1_reward"][t] and bool(d[0]) == bool(g["cfg1_done"][t])
        if bool(d[0]):
            env.reset()


def _oracle_batch(oracle, n, **kw):
    return oracle.BatchEnv(n, nthreads=8, **kw)


@pytest.mark.parametrize("flag", [0, 1])
def test_env_cw_batched_vs_oracle(golden, oracle, eng, flag):
    """2048 envs x 160 steps, random fp32 actions, short episodes + large capture radius so that captures,
    time-outs, auto-reset and the int64-truncation quirk all occur. Oracle = pinned C restatement."""
    g = golden("env_golden.npz")
    n, T = 2048, 160
    kw = dict(d_capture=181200.0, max_episode_steps=40, flag=flag)
    env = eng.EnvBatch(n, mode="cw", auto_reset=True, stm=g["stm100_columns"], **kw)
    orc = _oracle_batch(oracle, n, M=g["stm100_columns"], **kw)
    rng = np.random.default_rng(100 + flag)
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    n_done = 0
    n_eval = 0
    dz_mismatch_envs = np.zeros(n, dtype=bool)
    for t in range(T):
        pa = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        ea = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        r, d = env.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f64=obs)
        o_obs, o_r, o_d = orc.step(pa.astype(np.float64), ea.astype(np.float64))
        dz = env.dangerous_zone.cpu().numpy()
        o_dz = orc.aux()[3]
        dz_mismatch_envs |= (dz != o_dz)
        ok = ~dz_mismatch_envs
        # every env whose danger-zone history agrees must agree bit for bit in everything else
        assert np.array_equal(d.cpu().numpy()[ok], o_d[ok]), t
        assert np.array_equal(obs.cpu().numpy()[ok], o_obs[ok]), t
        assert np.array_equal(r.cpu().numpy()[ok], o_r[ok]), t
        n_done += int(o_d.sum())
        n_eval += int((~o_d.astype(bool)).sum())
    assert n_done > 1000                       # the episode-end paths really ran
    # The integer danger-zone count depends on the last bit of sin/cos/acos/atan/pow (fsolve's forward-difference
    # Jacobian at the +-pi/2 guesses amplifies one ulp into another root branch). The device therefore runs glibc's own
    # arithmetic (csrc/glibm.cuh): ZERO flips against the oracle (round 1, with libdevice: 2e-5 per evaluation).
    assert n_eval > 100000
    assert dz_mismatch_envs.sum() == 0, (int(dz_mismatch_envs.sum()), n_eval)
    assert int(env.err.sum()) == 0


def test_env_fast_libm_mode_is_the_documented_approximation(golden, oracle, eng):
    """SatEnvParams.fast_libm = 1 (opt-in): libdevice sin/cos/acos/atan and x*x instead of the host libm's arithmetic. Everything
    except the ill-conditioned danger-zone count stays bit-identical; the count may differ on ~3e-5 of the evaluations
    (bound here: 2e-4), and every env whose count history agrees is still bit-identical in obs / reward / done."""
    g = golden("env_golden.npz")
    n, T = 4096, 60
    kw = dict(d_capture=181200.0, max_episode_steps=40, flag=0)
    env = eng.EnvBatch(n, mode="cw", auto_reset=True, stm=g["stm100_columns"], fast_libm=True, **kw)
    orc = _oracle_batch(oracle, n, M=g["stm100_columns"], **kw)
    rng = np.random.default_rng(321)
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    flipped = np.zeros(n, dtype=bool)
    n_eval = 0
    for t in range(T):
        pa = rng.uniform(-2, 2, (n, 3)).astype(np.float32); ea = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        r, d = env.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f64=obs)
        o_obs, o_r, o_d = orc.step(pa.astype(np.float64), ea.astype(np.float64))
        flipped |= env.dangerous_zone.cpu().numpy() != orc.aux()[3]
        ok = ~flipped
        assert np.array_equal(d.cpu().numpy()[ok], o_d[ok]) and np.array_equal(r.cpu().numpy()[ok], o_r[ok])
        assert np.array_equal(obs.cpu().numpy()[ok], o_obs[ok])
        n_eval += int((~o_d.astype(bool)).sum())
    assert flipped.sum() <= 2e-4 * n_eval, (int(flipped.sum()), n_eval)


def test_danger_zone_counts_vs_reference_golden(golden, eng):
    """2997 states with the reference's own counts (Time_window_of_danger_zone...calculate_number_of_hanger_area)."""
    g = golden("danger_golden.npz")
    out = eng.danger_zone_count(torch.from_numpy(g["dz_states"]).cuda(), torch.from_numpy(g["dz_fuel"]).cuda())
    bad = int((out.cpu().numpy() != g["dz_count"]).sum())
    print(f"danger-zone counts differing from the reference's own: {bad} of {len(g['dz_count'])}")
    assert bad == 0, bad


def test_orbital_elements_bit_identical_to_oracle(oracle, eng):
    """calculate_orbital_elements (satellite_function.py:161-255) on 100 000 random near-GEO states: all six elements bit for
    bit (acos through the device libm, v_norm ** 2 through the device pow; the element a is a 1-ulp detector for the latter)."""
    from ppo_rl_satellite_b200 import _lib as L
    rng = np.random.default_rng(0)
    n = 100000
    rv = np.concatenate([np.array([27098000.0, 32306000.0, 0.0]) + rng.normal(0, 1e5, (n, 3)),
                         np.array([-2350.0, 1970.0, 0.0]) + rng.normal(0, 20, (n, 3))], axis=1)
    d_rv = torch.from_numpy(rv).cuda()
    out = torch.empty_like(d_rv)
    kind = torch.empty(n, dtype=torch.int32, device="cuda")
    L.check(L.load().sat_orbital_elements(d_rv.data_ptr(), n, 3.986e14, out.data_ptr(), kind.data_ptr(), L.stream_ptr()), "elements")
    want = np.array([oracle.orbital_elements(3.986e14, rv[i, 0:3], rv[i, 3:6])[:6] for i in range(n)])
    bad = (out.cpu().numpy().view(np.int64) != want.view(np.int64)).sum(axis=0)
    assert bad.sum() == 0, bad


def test_fsolve_roots_bit_identical_to_reference_golden(golden, eng):
    """The 4000 Numerical_iteration_method calls recorded from the reference (scipy.optimize.fsolve roots,
    satellite_function.py:558-565) through the DEVICE hybrd + device libm: every root bit for bit."""
    g = golden("danger_golden.npz")
    dev = lambda k: torch.from_numpy(g[k]).cuda()
    root, nfev = eng.numerical_iteration(dev("fs_dvm"), dev("fs_theta"), dev("fs_v1x"), dev("fs_v1y"), dev("fs_h"),
                                         dev("fs_guess"), u=3.986e14, return_nfev=True)
    got = root.cpu().numpy()
    bad = int((got.view(np.int64) != g["fs_root"].view(np.int64)).sum())
    print(f"fsolve roots differing from scipy's: {bad} of {len(got)}; evaluations per solve "
          f"{nfev.float().mean().item():.2f} (max {int(nfev.max())})")
    assert bad == 0, bad


@pytest.mark.parametrize("fn", ["sin", "cos", "sincos_s", "sincos_c", "acos", "atan", "pow2"])
def test_device_libm_bit_identical_to_host_libm(eng, fn):
    """csrc/glibm.cuh as compiled by nvcc for sm_100a vs the host libm the reference's numpy/python calls end in
    (python's math module calls libm directly; numpy scalar sin/cos do the same)."""
    import ctypes
    import math
    ver = ctypes.CDLL(None).gnu_get_libc_version
    ver.restype = ctypes.c_char_p
    if not ver().decode().startswith("2.39"):
        pytest.skip("glibm.cuh restates glibc 2.39")
    rng = np.random.default_rng(5)
    n = 60000
    if fn in ("sin", "cos", "sincos_s", "sincos_c"):
        x = np.concatenate([rng.uniform(-4, 4, n), rng.uniform(-200, 200, n), np.exp2(rng.uniform(-40, 26, n)) * rng.choice([-1, 1], n),
                            rng.integers(-1000, 1000, n) * (np.pi / 2) * (1 + rng.uniform(-1e-9, 1e-9, n)), [0.0, -0.0, 1e-300, 0.126, 0.855469, 2.426265]])
        ref = math.sin if fn in ("sin", "sincos_s") else math.cos
    elif fn == "acos":
        x = np.concatenate([rng.uniform(-1, 1, 2 * n), rng.choice([-1, 1], n) * (1 - np.exp2(-53 * rng.uniform(0, 1, n))), np.exp2(rng.uniform(-60, -2, n)),
                            [0.0, 1.0, -1.0, 0.125, 0.25, 0.5, 0.75, 0.921875, 0.953125, 0.96875]])
        ref = math.acos
    elif fn == "atan":
        x = np.concatenate([np.exp2(rng.uniform(-40, 60, 2 * n)) * rng.choice([-1, 1], 2 * n), rng.uniform(-20, 20, n), [0.0, -0.0, 1.0, 16.0, 0.0625, 1e300, -1e300]])
        ref = math.atan
    else:
        x = np.concatenate([np.exp2(rng.uniform(-360, 360, 2 * n)) * rng.choice([-1, 1], 2 * n), rng.uniform(-2, 2, n), 1 + rng.uniform(-1e-9, 1e-9, n), [0.0, 1.0, -1.0, 2.0]])
        ref = lambda v: math.pow(v, 2.0)
    got = eng.libm_eval(fn, torch.from_numpy(x).cuda()).cpu().numpy()
    want = np.array([ref(float(v)) for v in x])
    bad = int((got.view(np.int64) != want.view(np.int64)).sum())
    assert bad == 0, (fn, bad, len(x))


def test_env_ragged_and_tiny_batches(golden, oracle, eng):
    g = golden("env_golden.npz")
    for n in (1, 2, 31, 33, 65):
        env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=5, stm=g["stm100_columns"])
        orc = _oracle_batch(oracle, n, M=g["stm100_columns"], d_capture=20000.0, max_episode_steps=5)
        rng = np.random.default_rng(n)
        obs = torch.empty((n, 18), dtype=torch.float32, device="cuda")
        for t in range(12):
            pa = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
            ea = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
            r, d = env.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f32=obs)
            o_obs, o_r, o_d = orc.step(pa.astype(np.float64), ea.astype(np.float64))
            assert np.array_equal(d.cpu().numpy(), o_d)
            assert np.array_equal(r.cpu().numpy(), o_r)
            assert np.array_equal(obs.cpu().numpy(), o_obs.astype(np.float32))


def test_env_step_host_buffers(golden, oracle, eng):
    g = golden("env_golden.npz")
    n = 257
    env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=7, stm=g["stm100_columns"])
    orc = _oracle_batch(oracle, n, M=g["stm100_columns"], d_capture=20000.0, max_episode_steps=7)
    rng = np.random.default_rng(5)
    for t in range(10):
        pa = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        ea = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        obs, r, d = env.step_host(pa, ea, chunks=(1, 2, 4, 0, -2)[t % 5])                # single-range / pipelined / zero-copy forms
        o_obs, o_r, o_d = orc.step(pa.astype(np.float64), ea.astype(np.float64))
        assert np.array_equal(d, o_d) and np.array_equal(r, o_r) and np.array_equal(obs, o_obs.astype(np.float32))


def test_env_step_host_rk4_forms_equal_device_step(eng):
    """rk4 mode: every host-buffer form (overlapped observation copy = default, zero-copy ranges, staged) returns exactly
    what the device-resident step returns, including the observation after an auto reset (captures and time-outs occur)"""
    n = 1500
    rng = np.random.default_rng(11)
    kw = dict(mode="rk4", substeps=5, h=1.0, d_capture=150000.0, max_episode_steps=6)
    for chunks in (0, -2, -3, 1, 2):
        a, b = eng.EnvBatch(n, **kw), eng.EnvBatch(n, **kw)
        P0 = np.array([200000.0, 0, 0]) + rng.normal(0, 6e4, (n, 3)); E0 = np.array([18000.0, 0, 0]) + rng.normal(0, 6e4, (n, 3))
        V0 = rng.normal(0, 3.0, (n, 3)); W0 = rng.normal(0, 3.0, (n, 3))
        a.set_state(P0, V0, E0, W0); b.set_state(P0, V0, E0, W0)
        obs_d = torch.empty((n, 18), dtype=torch.float32, device="cuda")
        dones = 0
        for t in range(9):
            pa = rng.uniform(-2, 2, (n, 3)).astype(np.float32); ea = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
            r, d = a.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f32=obs_d)
            obs, rh, dh = b.step_host(pa, ea, chunks=chunks)
            assert np.array_equal(dh, d.cpu().numpy()) and np.array_equal(rh, r.cpu().numpy())
            assert np.array_equal(obs, obs_d.cpu().numpy())
            dones += int(dh.sum())
        assert dones > n                                       # every env timed out at least once, some were captured
        assert torch.equal(a.state, b.state) and torch.equal(a.istate, b.istate)


def test_env_argument_errors(eng):
    from ppo_rl_satellite_b200 import _lib as L
    import ctypes as C
    env = eng.EnvBatch(4)
    lib = L.load()
    a = torch.zeros((4, 3), dtype=torch.float32, device="cuda")
    rc = lib.sat_env_step(C.byref(env.st), a.data_ptr(), a.data_ptr(), None, None, None, None, None, None,
                          None, None, None, None, C.byref(env.params), None)
    assert rc == -1                                         # reward/done missing
    env.params.mode = 7
    rc = lib.sat_env_step(C.byref(env.st), a.data_ptr(), a.data_ptr(), None, None, None, None, env.reward.data_ptr(),
                          env.done.data_ptr(), None, None, None, None, C.byref(env.params), None)
    assert rc == -3
    with pytest.raises(L.SatError):
        env.step(a, a.double())


# ============================================================================ K2: rk4 mode
def test_env_rk4_mode_vs_oracle(oracle, eng):
    """rk4 mode has no upstream env; the oracle composes the reference's step logic with the script's RK4.
    States to 1e-9 relative (north star bar), rewards to 1e-6, dones identical; the danger-zone count may flip
    on the ill-conditioned states (see test_env_cw_batched_vs_oracle) because the integrators differ at 1e-15:
    envs whose count history differs are excluded from later comparisons (the count gates the next impulse)."""
    n, T, S = 512, 12, 20
    kw = dict(d_capture=20000.0, max_episode_steps=1000)
    env = eng.EnvBatch(n, mode="rk4", substeps=S, h=1.0, auto_reset=True, **kw)
    orc = _oracle_batch(oracle, n, **kw)
    rng = np.random.default_rng(3)
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    R = np.array([27098000.0, 32306000.0, 0.0]); V = np.array([-2350.0, 1970.0, 0.0])
    diverged = np.zeros(n, dtype=bool)
    for t in range(T):
        pa = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        ea = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        r, d = env.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f64=obs)
        o_obs, o_r, o_d = orc.step_rk4(pa.astype(np.float64), ea.astype(np.float64), h=1.0, substeps=S)
        dz_same = env.dangerous_zone.cpu().numpy() == orc.aux()[3]
        ok = ~diverged
        assert np.array_equal(d.cpu().numpy()[ok], o_d[ok])
        got = obs.cpu().numpy()
        # positions are ~1e5 m relative to an origin 4.2e7 m from the Earth's centre: compare in the inertial
        # frame the integrator works in
        for lo in (6, 12):
            dr = np.linalg.norm(got[ok, lo:lo + 3] - o_obs[ok, lo:lo + 3], axis=1) / np.linalg.norm(o_obs[ok, lo:lo + 3] + R, axis=1)
            dv = np.linalg.norm(got[ok, lo + 3:lo + 6] - o_obs[ok, lo + 3:lo + 6], axis=1) / np.linalg.norm(o_obs[ok, lo + 3:lo + 6] + V, axis=1)
            assert dr.max() < 1e-9 and dv.max() < 1e-9, (t, dr.max(), dv.max())
        both = ok & dz_same
        np.testing.assert_allclose(r.cpu().numpy()[both], o_r[both], rtol=0, atol=1e-6)
        diverged |= ~dz_same
    assert diverged.mean() < 0.02, diverged.mean()


# ============================================================================ normalisation
def test_normalization_n1_sequence_is_the_reference(golden, eng):
    g = golden("norm_golden.npz")
    rs = eng.RunningStats(18)
    X = torch.from_numpy(g["x"]).cuda()
    for k in range(X.shape[0]):
        out = rs.update_normalize(X[k:k + 1])
        assert np.array_equal(out.cpu().numpy()[0], g["x_normed"][k]), k
    assert rs.n == int(g["final_n"])
    assert np.array_equal(rs.mean.cpu().numpy(), g["final_mean"])
    assert np.array_equal(rs.S.cpu().numpy(), g["final_S"])
    assert np.array_equal(rs.std.cpu().numpy(), g["final_std"])


def test_normalization_batched_matches_chan_merge(golden, oracle, eng):
    g = golden("env_golden.npz")
    X = g["long_obs"]
    rs = eng.RunningStats(18)
    n, mean, S = 0, np.zeros(18), np.zeros(18)
    for lo in range(0, 3000, 500):
        xb = X[lo:lo + 500]
        out = rs.update_normalize(torch.from_numpy(xb).cuda())
        n, mean, S = oracle.chan_merge(n, mean, S, xb)
        std = np.sqrt(S / n)
        np.testing.assert_allclose(rs.mean.cpu().numpy(), mean, rtol=1e-13, atol=1e-9)
        np.testing.assert_allclose(rs.S.cpu().numpy(), S, rtol=1e-11, atol=1e-6)
        np.testing.assert_allclose(out.cpu().numpy(), (xb - mean) / (std + 1e-8), rtol=1e-9, atol=1e-9)
    assert rs.n == 3000
    frozen = rs.update_normalize(torch.from_numpy(X[:7]).cuda(), update=False)
    assert rs.n == 3000 and frozen.shape == (7, 18)


def test_env_fused_running_stats(golden, oracle, eng):
    """obs / discounted-return statistics updated inside the env step equal a Chan merge of the same batches."""
    g = golden("env_golden.npz")
    n = 300
    env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=9, stm=g["stm100_columns"], gamma=0.99)
    obs_stats, ret_stats = eng.RunningStats(18), eng.RunningStats(1)
    std_out = torch.zeros(1, dtype=torch.float64, device="cuda")
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    rng = np.random.default_rng(8)
    cnt, mean, S = 0, np.zeros(18), np.zeros(18)
    rc, rmean, rS = 0, np.zeros(1), np.zeros(1)
    R = np.zeros(n)
    for t in range(25):
        pa = torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda()
        ea = torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda()
        r, d = env.step(pa, ea, obs_f64=obs, obs_stats=obs_stats, ret_stats=ret_stats, ret_std_out=std_out)
        cnt, mean, S = oracle.chan_merge(cnt, mean, S, obs.cpu().numpy())
        R = 0.99 * R + r.cpu().numpy()
        rc, rmean, rS = oracle.chan_merge(rc, rmean, rS, R[:, None])
        R[d.cpu().numpy() > 0] = 0.0
        np.testing.assert_allclose(obs_stats.mean.cpu().numpy(), mean, rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(obs_stats.S.cpu().numpy(), S, rtol=1e-10, atol=1e-5)
        np.testing.assert_allclose(ret_stats.S.cpu().numpy(), rS, rtol=1e-10, atol=1e-8)
        np.testing.assert_allclose(float(std_out[0]), np.sqrt(rS[0] / rc), rtol=1e-12)
    assert obs_stats.n == 25 * n and ret_stats.n == 25 * n
    np.testing.assert_allclose(env.state[15].cpu().numpy(), R, rtol=1e-13, atol=1e-12)


# ============================================================================ K4: GAE
def test_gae_flat_bit_identical_to_reference_block(golden, eng):
    g = golden("ppo_golden.npz")
    c = lambda k: torch.from_numpy(g[k]).cuda()
    adv, vt = eng.gae_flat(c("gae_r"), c("gae_vs"), c("gae_vs_next"), c("gae_done"), c("gae_done"))
    assert np.array_equal(adv.cpu().numpy(), g["gae_adv"])         # bar is 1e-6; the kernel is exact
    assert np.array_equal(vt.cpu().numpy(), g["gae_v_target"])
    eng.adv_normalize_(adv, group=False)
    np.testing.assert_allclose(adv.cpu().numpy(), g["gae_adv_normed"], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("T,N", [(1, 1), (7, 3), (256, 1000), (2048, 64)])
def test_gae_time_major_vs_oracle(oracle, eng, T, N):
    rng = np.random.default_rng(T * 131 + N)
    r = rng.normal(0, 2, (T, N)).astype(np.float32)
    v = rng.normal(0, 5, (T + 1, N)).astype(np.float32)
    done = (rng.random((T, N)) < 0.03).astype(np.uint8)
    adv, vt = eng.gae_time_major(torch.from_numpy(r).cuda(), torch.from_numpy(v).cuda(), torch.from_numpy(done).cuda())
    o_adv, o_vt = oracle.gae_time_major(r, v, done)
    assert np.array_equal(adv.cpu().numpy(), o_adv) and np.array_equal(vt.cpu().numpy(), o_vt)


def test_gae_reward_scale_and_chunked_flat(oracle, eng):
    rng = np.random.default_rng(4)
    T, N = 50, 10
    r = rng.normal(0, 2, (T, N)).astype(np.float32)
    v = rng.normal(0, 5, (T + 1, N)).astype(np.float32)
    done = (rng.random((T, N)) < 0.1).astype(np.uint8)
    sc = rng.uniform(0.1, 2.0, T).astype(np.float32)
    adv, _ = eng.gae_time_major(torch.from_numpy(r).cuda(), torch.from_numpy(v).cuda(), torch.from_numpy(done).cuda(),
                                r_scale=torch.from_numpy(sc).cuda())
    o_adv, _ = oracle.gae_time_major(r * sc[:, None], v, done)
    assert np.array_equal(adv.cpu().numpy(), o_adv)
    B = 10000                                               # > one shared-memory chunk
    r1 = rng.normal(0, 1, B).astype(np.float32); vs = rng.normal(0, 1, B).astype(np.float32)
    vn = rng.normal(0, 1, B).astype(np.float32); dn = (rng.random(B) < 0.01).astype(np.float32)
    c = lambda a: torch.from_numpy(a).cuda()
    a2, t2 = eng.gae_flat(c(r1), c(vs), c(vn), c(dn), c(dn))
    oa, ot = oracle.gae(r1, vs, vn, dn, dn)
    assert np.array_equal(a2.cpu().numpy(), oa) and np.array_equal(t2.cpu().numpy(), ot)


# ============================================================================ K3: actor / critic
def _weights(g, prefix):
    return {k[len(prefix):]: g[k] for k in g.files if k.startswith(prefix)}


def test_actor_matches_reference_outputs(golden, eng):
    g = golden("ppo_golden.npz")
    actor = eng.GaussianActorKernel(max_action=1.6).load_state_dict(_weights(g, "actor."))
    obs = torch.from_numpy(g["obs"]).cuda()
    n = obs.shape[0]
    mean = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    act, logp = actor.sample(obs=obs, eps_in=torch.from_numpy(g["eps"]).cuda(), mean_out=mean)
    m = mean.cpu().numpy()
    # rows [0,384): raw env-scale observations (pre-activations ~1e5 in fp32); rows [384,768): unit scale
    np.testing.assert_allclose(m[:384], g["mean"][:384], rtol=0, atol=1e-4)
    np.testing.assert_allclose(m[384:], g["mean"][384:], rtol=0, atol=2e-5)
    np.testing.assert_allclose(act.cpu().numpy()[384:], g["action"][384:], rtol=0, atol=2e-5)
    np.testing.assert_allclose(logp.cpu().numpy()[384:], g["logp"][384:], rtol=1e-4, atol=1e-4)


def test_critic_matches_reference_outputs(golden, eng):
    g = golden("ppo_golden.npz")
    critic = eng.GaussianActorKernel(critic=True).load_state_dict(_weights(g, "critic."))
    v = critic.value(torch.from_numpy(g["obs"]).cuda())
    np.testing.assert_allclose(v.cpu().numpy()[384:], g["value"][384:], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(v.cpu().numpy()[:384], g["value"][:384], rtol=1e-3, atol=1e-3)


def test_actor_vs_oracle_ragged(golden, oracle, eng):
    g = golden("ppo_golden.npz")
    W = _weights(g, "actor.")
    actor = eng.GaussianActorKernel().load_state_dict(W)
    rng = np.random.default_rng(2)
    for n in (1, 63, 64, 65, 1000):
        obs = rng.normal(0, 1, (n, 18)).astype(np.float32)
        eps = rng.normal(0, 1, (n, 3)).astype(np.float32)
        mean = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        act, logp = actor.sample(obs=torch.from_numpy(obs).cuda(), eps_in=torch.from_numpy(eps).cuda(), mean_out=mean)
        o_mean = oracle.actor_forward(W, obs)
        o_a, o_lp = oracle.gaussian_sample(mean.cpu().numpy(), W["log_std"], eps)
        np.testing.assert_allclose(mean.cpu().numpy(), o_mean, rtol=0, atol=2e-5)
        np.testing.assert_allclose(act.cpu().numpy(), o_a, rtol=0, atol=1e-6)
        np.testing.assert_allclose(logp.cpu().numpy(), o_lp, rtol=1e-5, atol=1e-5)


def test_actor_philox_sampling_properties(golden, eng):
    g = golden("ppo_golden.npz")
    actor = eng.GaussianActorKernel().load_state_dict(_weights(g, "actor."))
    n = 1 << 17
    obs = torch.zeros((n, 18), dtype=torch.float32, device="cuda")
    eps = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    a1, _ = actor.sample(obs=obs, seed=7, step=3, eps_out=eps)
    e = eps.cpu().numpy().astype(np.float64)
    assert abs(e.mean()) < 0.01 and abs(e.var() - 1.0) < 0.02
    assert abs((e ** 3).mean()) < 0.03 and abs((e ** 4).mean() - 3.0) < 0.1
    assert abs(np.corrcoef(e[:, 0], e[:, 1])[0, 1]) < 0.01
    a2, _ = actor.sample(obs=obs, seed=7, step=3)
    assert torch.equal(a1, a2)                                # reproducible
    a3, _ = actor.sample(obs=obs, seed=7, step=4)
    assert not torch.equal(a1, a3)
    # shard invariance: rows [k, n) computed as a separate shard with row_offset = k give the same draws
    k = 1000
    a4, _ = actor.sample(obs=obs[k:], seed=7, step=3, row_offset=k)
    assert torch.equal(a1[k:], a4)


def test_actor_fused_state_path_equals_observe_path(golden, eng):
    g = golden("ppo_golden.npz")
    actor = eng.GaussianActorKernel().load_state_dict(_weights(g, "actor."))
    n = 500
    env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=50)
    rng = np.random.default_rng(0)
    stats = eng.RunningStats(18)
    for t in range(5):
        env.step(torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda(),
                 torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda(), obs_stats=stats)
    eps = torch.from_numpy(rng.normal(0, 1, (n, 3)).astype(np.float32)).cuda()
    obs_out = torch.empty((n, 18), dtype=torch.float32, device="cuda")
    a_f, lp_f = actor.sample(env=env, obs_stats=stats, eps_in=eps, obs_out=obs_out)
    x = env.observe()
    xn = ((x - stats.mean) / (stats.std + 1e-8)).float()
    assert torch.equal(obs_out, xn)
    a_o, lp_o = actor.sample(obs=xn, eps_in=eps)
    assert torch.equal(a_f, a_o) and torch.equal(lp_f, lp_o)


# ============================================================================ sharding / resume
def test_env_shard_invariance_emulated_ranks(golden, eng):
    """config 4 shape in miniature: splitting the env axis over ranks changes nothing per env (ranks emulated as
    separate batches on one GPU; there is no cross-env term and no collective in the rollout)."""
    g = golden("env_golden.npz")
    n, T = 1024, 12
    kw = dict(mode="rk4", substeps=7, h=1.0, d_capture=20000.0, max_episode_steps=5)
    full = eng.EnvBatch(n, **kw)
    shards = [eng.EnvBatch(n // 4, **kw) for _ in range(4)]
    rng = np.random.default_rng(0)
    for t in range(T):
        pa = torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda()
        ea = torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda()
        r, d = full.step(pa, ea)
        for k, sh in enumerate(shards):
            lo, hi = k * n // 4, (k + 1) * n // 4
            rs, ds = sh.step(pa[lo:hi].contiguous(), ea[lo:hi].contiguous())
            assert torch.equal(rs, r[lo:hi]) and torch.equal(ds, d[lo:hi])
            assert torch.equal(sh.state, full.state[:, lo:hi]) and torch.equal(sh.istate, full.istate[:, lo:hi])


def test_env_checkpoint_resume_is_exact(eng):
    n = 300
    kw = dict(mode="cw", d_capture=20000.0, max_episode_steps=6)
    a = eng.EnvBatch(n, **kw)
    rng = np.random.default_rng(1)
    acts = [(torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda(),
             torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda()) for _ in range(10)]
    for pa, ea in acts[:5]:
        a.step(pa, ea)
    sd = a.state_dict()
    b = eng.EnvBatch(n, **kw).load_state_dict(sd)
    for pa, ea in acts[5:]:
        ra, da = a.step(pa, ea)
        rb, db = b.step(pa, ea)
        assert torch.equal(ra, rb) and torch.equal(da, db)
    assert torch.equal(a.state, b.state) and torch.equal(a.istate, b.istate)


# ============================================================================ BASELINE full sizes: size-independent properties
def test_full_size_rk4_conservation_and_time_reversal(eng):
    """1 048 576 random LEO/GEO states (config 4 size) x 1000 steps: energy and angular momentum are conserved with J2
    off, and integrating back with -h returns to the start (RK4 is not symmetric: the residual is its truncation error)."""
    n = 1 << 20
    g = torch.Generator(device="cuda").manual_seed(0)
    r = torch.where(torch.arange(n, device="cuda") % 2 == 0, 6778.0 + 600.0 * torch.rand(n, generator=g, device="cuda", dtype=torch.float64),
                    42164.0 + 100.0 * (torch.rand(n, generator=g, device="cuda", dtype=torch.float64) - 0.5))
    ang = 6.283185307179586 * torch.rand(n, generator=g, device="cuda", dtype=torch.float64)
    inc = 1.5 * torch.rand(n, generator=g, device="cuda", dtype=torch.float64)
    v = torch.sqrt(398600.0 / r) * (1.0 + 0.01 * (torch.rand(n, generator=g, device="cuda", dtype=torch.float64) - 0.5))
    x, _ = eng.alloc_soa(6, n, torch.float64, "cuda")
    x[0], x[1], x[2] = r * torch.cos(ang), r * torch.sin(ang) * torch.cos(inc), r * torch.sin(ang) * torch.sin(inc)
    x[3], x[4], x[5] = -v * torch.sin(ang), v * torch.cos(ang) * torch.cos(inc), v * torch.cos(ang) * torch.sin(inc)
    x0 = x.clone()

    def energy(s):
        return 0.5 * (s[3:] ** 2).sum(0) - 398600.0 / torch.linalg.norm(s[:3], dim=0)

    def hvec(s):
        return torch.linalg.cross(s[:3].T, s[3:].T)
    eng.rk4_propagate(x, 1.0, 1000, j2=0.0)
    assert float((energy(x) / energy(x0) - 1).abs().max()) < 1e-10
    assert float((torch.linalg.norm(hvec(x) - hvec(x0), dim=1) / torch.linalg.norm(hvec(x0), dim=1)).max()) < 1e-12
    eng.rk4_propagate(x, -1.0, 1000, j2=0.0)
    back = float((torch.linalg.norm(x[:3] - x0[:3], dim=0) / torch.linalg.norm(x0[:3], dim=0)).max())
    assert back < 1e-9, back
    # with J2 on, the z component of angular momentum is still conserved (axial symmetry)
    eng.rk4_propagate(x, 1.0, 1000)
    assert float(((hvec(x)[:, 2] - hvec(x0)[:, 2]).abs() / torch.linalg.norm(hvec(x0), dim=1)).max()) < 1e-9


def test_full_size_env_batch_subset_vs_oracle(golden, oracle, eng):
    """config 3 size (65 536 envs, cw mode): a random subset of 1024 envs is stepped by the oracle with the same actions and
    must agree bit for bit (envs are independent), danger-zone counts included."""
    g = golden("env_golden.npz")
    n, m, T = 65536, 1024, 24
    kw = dict(d_capture=181200.0, max_episode_steps=10)
    env = eng.EnvBatch(n, mode="cw", auto_reset=True, stm=g["stm100_columns"], **kw)
    rng = np.random.default_rng(7)
    sub = np.sort(rng.choice(n, m, replace=False))
    orc = _oracle_batch(oracle, m, M=g["stm100_columns"], **kw)
    obs = torch.empty((n, 18), dtype=torch.float64, device="cuda")
    flipped = np.zeros(m, dtype=bool)
    for t in range(T):
        pa = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        ea = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
        r, d = env.step(torch.from_numpy(pa).cuda(), torch.from_numpy(ea).cuda(), obs_f64=obs)
        o_obs, o_r, o_d = orc.step(pa[sub].astype(np.float64), ea[sub].astype(np.float64))
        flipped |= env.dangerous_zone.cpu().numpy()[sub] != orc.aux()[3]
        ok = ~flipped
        assert np.array_equal(d.cpu().numpy()[sub][ok], o_d[ok])
        assert np.array_equal(r.cpu().numpy()[sub][ok], o_r[ok])
        assert np.array_equal(obs.cpu().numpy()[sub][ok], o_obs[ok])
    assert flipped.sum() == 0, int(flipped.sum())
    assert int(env.err.sum()) == 0 and int(env.done.sum()) >= 0


def test_empty_and_invalid_sizes_return_error_codes(eng):
    """empty inputs are argument errors (SAT_ERR_SIZE = -2), never a launch"""
    from ppo_rl_satellite_b200 import _lib as L
    import ctypes as C
    lib = L.load()
    x = torch.zeros(64, dtype=torch.float64, device="cuda")
    i32 = torch.zeros(64, dtype=torch.int32, device="cuda")
    f32 = torch.zeros(64, dtype=torch.float32, device="cuda")
    u8 = torch.zeros(64, dtype=torch.uint8, device="cuda")
    st = L.SatEnvState(x.data_ptr(), i32.data_ptr(), 0, 0)
    p = L.default_params()
    assert lib.sat_env_init(C.byref(st), 320.0, 320.0, C.byref(p), None) == -2
    assert lib.sat_env_step(C.byref(st), f32.data_ptr(), f32.data_ptr(), None, None, None, None, x.data_ptr(), u8.data_ptr(),
                            None, None, None, None, C.byref(p), None) == -2
    st_odd = L.SatEnvState(x.data_ptr(), i32.data_ptr(), 3, 3)            # ld must be even
    assert lib.sat_env_observe(C.byref(st_odd), f32.data_ptr(), None, None) == -2
    assert lib.sat_gae(f32.data_ptr(), f32.data_ptr(), u8.data_ptr(), None, 0, 4, 0.99, 0.95, f32.data_ptr(), f32.data_ptr(), None) == -2
    assert lib.sat_gae_flat(f32.data_ptr(), f32.data_ptr(), f32.data_ptr(), f32.data_ptr(), f32.data_ptr(), 0, 0.99, 0.95,
                            f32.data_ptr(), f32.data_ptr(), None) == -2
    assert lib.sat_norm_update(x.data_ptr(), x.data_ptr(), 0, 18, 1, None, None, x.data_ptr(), None) == -2
    assert lib.sat_norm_update(x.data_ptr(), x.data_ptr(), 4, 33, 1, None, None, x.data_ptr(), None) == -2   # dim > 32
    assert lib.sat_danger_zone_count(x.data_ptr(), x.data_ptr(), 0, 3.986e14, i32.data_ptr(), None, None) == -2
    assert lib.sat_cw_ode_rk45(x.data_ptr(), 4, 4, -1.0, 1.0, 1.0, 1.0, 1e-3, 1e-6, None, None) == -2
    w = L.SatActorWeights()
    assert lib.sat_actor_sample(C.byref(w), f32.data_ptr(), None, None, 4, 0, 0, 0, None, f32.data_ptr(), f32.data_ptr(),
                                None, None, None, None) == -1            # weights not packed
    with pytest.raises(L.SatError):
        eng.EnvBatch(0)


def test_actor_relu_and_max_action_variants_vs_torch(eng):
    """args.use_tanh = 0 (ReLU hidden activations, ppo_continuous.py:74) and a non-default max_action, against torch fp32"""
    torch.manual_seed(3)
    W = {"fc1.weight": torch.randn(256, 18) * 0.3, "fc1.bias": torch.randn(256) * 0.1, "fc2.weight": torch.randn(256, 256) * 0.08,
         "fc2.bias": torch.randn(256) * 0.1, "mean_layer.weight": torch.randn(3, 256) * 0.05, "mean_layer.bias": torch.randn(3) * 0.1,
         "log_std": torch.tensor([[-0.5, 0.0, 0.3]])}
    x = torch.randn(777, 18)
    eps = torch.randn(777, 3)
    for use_tanh, max_action in ((False, 1.6), (True, 0.4)):
        act_fn = torch.tanh if use_tanh else torch.relu
        h = act_fn(act_fn(x @ W["fc1.weight"].T + W["fc1.bias"]) @ W["fc2.weight"].T + W["fc2.bias"])
        mean_ref = max_action * torch.tanh(h @ W["mean_layer.weight"].T + W["mean_layer.bias"])
        std = torch.exp(W["log_std"])
        a_ref = torch.clamp(mean_ref + std * eps, -max_action, max_action)
        lp_ref = torch.distributions.Normal(mean_ref, std.expand_as(mean_ref)).log_prob(a_ref)
        k = eng.GaussianActorKernel(max_action=max_action, use_tanh=use_tanh).load_state_dict(W)
        mean = torch.empty(777, 3, device="cuda")
        a, lp = k.sample(obs=x.cuda(), eps_in=eps.cuda(), mean_out=mean)
        torch.testing.assert_close(mean.cpu(), mean_ref, rtol=0, atol=3e-5)
        torch.testing.assert_close(a.cpu(), a_ref, rtol=0, atol=3e-5)
        torch.testing.assert_close(lp.cpu(), lp_ref, rtol=1e-4, atol=2e-4)


# ============================================================================ reachable-domain sweep (s8 f.3)
def test_reachable_domain_sweep_vs_reference_and_oracle(golden, oracle, eng):
    g = golden("reach_golden.npz")
    N = int(g["N"])
    hi, lo, valid = eng.reachable_domain(torch.from_numpy(g["elements"]).cuda(), torch.from_numpy(g["delta_max"]).cuda(), N, N)
    hi, lo, valid = hi.cpu().numpy(), lo.cpu().numpy(), valid.cpu().numpy().astype(bool)
    for n in range(len(g["idx"])):
        assert valid[n].sum() == len(g[f"rf_max_{n}"])               # same directions pass the reachability test
        np.testing.assert_allclose(hi[n][valid[n]], g[f"rf_max_{n}"], rtol=1e-9, atol=1e-3)
        np.testing.assert_allclose(lo[n][valid[n]], g[f"rf_min_{n}"], rtol=1e-9, atol=1e-3)
    # full 201 x 201 sweep (the reference's N2 = N3 = 200) for two states against the oracle
    for n in (0, 3):
        h2, l2, v2 = eng.reachable_domain(torch.from_numpy(g["elements"][n:n + 1]).cuda(), torch.from_numpy(g["delta_max"][n:n + 1]).cuda())
        oh, ol, ov = oracle.reachable_domain(g["elements"][n], g["delta_max"][n], 200, 200)
        v2 = v2.cpu().numpy()[0].astype(bool)
        assert np.array_equal(v2, ov)
        np.testing.assert_allclose(h2.cpu().numpy()[0][v2], oh, rtol=1e-9, atol=1e-3)
        np.testing.assert_allclose(l2.cpu().numpy()[0][v2], ol, rtol=1e-9, atol=1e-3)


def test_step_timed_is_the_same_step(eng):
    """sat_env_step_timed (bench.py's per-launch timing) runs exactly the launches of sat_env_step"""
    n = 1000
    rng = np.random.default_rng(5)
    kw = dict(mode="rk4", substeps=10, h=1.0, d_capture=20000.0, max_episode_steps=50)
    a, b = eng.EnvBatch(n, **kw), eng.EnvBatch(n, **kw)
    for t in range(3):
        pa = torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda()
        ea = torch.from_numpy(rng.uniform(-2, 2, (n, 3)).astype(np.float32)).cuda()
        ra, da = a.step(pa, ea)
        ms = b.step_timed(pa, ea)
        assert len(ms) == 3 and ms[0] > 0 and ms[1] > 0
        assert torch.equal(ra, b.reward) and torch.equal(da, b.done)
    assert torch.equal(a.state, b.state) and torch.equal(a.istate, b.istate)


@pytest.mark.parametrize("tc", [False, True])
def test_actor_sample_pair_equals_two_calls(golden, eng, tc):
    """sat_actor_sample_pair / sat_actor_sample_pair_tc: both networks in one launch, bit-identical to two single calls"""
    g = golden("ppo_golden.npz")
    W = _weights(g, "actor.")
    a = eng.GaussianActorKernel().load_state_dict(W)
    W2 = {k: (v * 0.9 + 0.01) for k, v in W.items()}
    b = eng.GaussianActorKernel().load_state_dict(W2)
    for n in (1, 63, 1000, 20000):
        env = eng.EnvBatch(n, mode="cw")
        rng = np.random.default_rng(n)
        env.set_state(np.array([2e5, 0, 0]) + rng.normal(0, 3e4, (n, 3)), rng.normal(0, 3, (n, 3)),
                      np.array([1.8e4, 0, 0]) + rng.normal(0, 3e4, (n, 3)), rng.normal(0, 3, (n, 3)))
        stats = eng.RunningStats(18)
        stats.update_normalize(env.observe())
        obs1 = torch.empty((n, 18), dtype=torch.float32, device="cuda"); obs2 = torch.empty_like(obs1)
        a1, l1 = a.sample(env=env, obs_stats=stats, seed=3, step=10, row_offset=7, obs_out=obs1, tc=tc)
        b1, m1 = b.sample(env=env, obs_stats=stats, seed=3, step=11, row_offset=7, tc=tc)
        a2, l2, b2, m2 = a.sample_pair(b, env=env, obs_stats=stats, seed=3, step=10, other_step=11, row_offset=7, obs_out=obs2, tc=tc)
        for x, y in ((a1, a2), (l1, l2), (b1, b2), (m1, m2), (obs1, obs2)):
            assert torch.equal(x, y)
        assert not torch.equal(a1, b1)
