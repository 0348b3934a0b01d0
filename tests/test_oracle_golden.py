"""Pins the CPU oracle (oracle/sat_oracle.c) against fixtures produced by the reference itself
(tests/golden/make_golden.py) and against the reference's own known-answer data. CPU only."""
import numpy as np
import pytest


def rel_err_rv(x, y):
    dr = np.linalg.norm(x[:3] - y[:3], axis=0) / np.linalg.norm(y[:3], axis=0)
    dv = np.linalg.norm(x[3:] - y[3:], axis=0) / np.linalg.norm(y[3:], axis=0)
    return max(dr.max(), dv.max())


# ------------------------------------------------------------------ RK4 (script :15-40)
def test_state_eq_matches_reference(golden, oracle):
    g = golden("rk4_golden.npz")
    for p, f in zip(g["stateeq_in"], g["stateeq_out"]):
        np.testing.assert_allclose(oracle.state_eq(p), f, rtol=2e-15, atol=0)


@pytest.mark.parametrize("tag,j2", [("j2off", 0.0), ("j2on", 0.00108263)])
def test_rk4_1000_steps_config2(golden, oracle, tag, j2):
    g = golden("rk4_golden.npz")
    x = oracle.rk4_propagate(g["x0"], 1.0, 1000, j2=j2, nthreads=8)
    # reference RungeKutta on the (6, 4096) array; bar is 1e-9, the literal restatement sits at ~1e-15
    assert rel_err_rv(x, g[f"x1000_{tag}"]) < 5e-14
    # scalar path as shipped (one state per call)
    idx = g["scalar_idx"]
    assert rel_err_rv(x[:, idx], g[f"x1000_scalar_{tag}"]) < 5e-14


def test_rk4_script_initial_condition_86400(golden, oracle):
    g = golden("rk4_golden.npz")
    x = oracle.rk4_propagate(g["script_ic"].reshape(6, 1), 1.0, 86400)
    ref = g["script_86400"].reshape(6, 1)
    # SURVEY.md s6 regression vector (what the script prints)
    survey = np.array([6455.3427883148706, 1813.7238301483098, 1514.2847686660500,
                       -2.4403782721782639, 3.3699366990985862, 6.3867370933957881]).reshape(6, 1)
    assert rel_err_rv(ref, survey) < 1e-15
    assert rel_err_rv(x, ref) < 1e-11


# ------------------------------------------------------------------ elements (satellite_function.py:161-315)
def test_orbital_elements_known_answer_841(golden, oracle):
    g = golden("elements_golden.npz")
    csv = g["csv_a_e_i_f_fuel"]
    for k in range(len(g["R"])):
        el = oracle.orbital_elements(3.986e14, g["R"][k], g["V"][k])
        assert len(el) == 6
        a, e, i, om, Om, f = el
        # the reference's own stored answers (a, e, i, f); tolerances from SURVEY.md s4 probe
        assert abs(a - csv[k, 0]) / csv[k, 0] < 1e-14
        assert abs(e - csv[k, 1]) < 1e-13
        assert abs(i - csv[k, 2]) < 1e-11
        assert abs(f - csv[k, 3]) < 1e-9 * max(1.0, abs(csv[k, 3]))
        np.testing.assert_allclose(el, g["elements_live"][k], rtol=1e-12, atol=1e-12)


def test_state_information_roundtrip(golden, oracle):
    g = golden("elements_golden.npz")
    for k in range(0, len(g["R"]), 7):
        R, V = oracle.state_information(g["elements_live"][k], 3.986e14)
        np.testing.assert_allclose(np.concatenate([R, V]), g["state_roundtrip"][k], rtol=1e-13, atol=1e-9)


# ------------------------------------------------------------------ fsolve / danger zone
def test_fsolve_roots_bit_identical(golden, oracle):
    g = golden("danger_golden.npz")
    n = len(g["fs_root"])
    got = np.array([oracle.numerical_iteration(3.986e14, g["fs_dvm"][k], g["fs_theta"][k], g["fs_v1x"][k],
                                               g["fs_v1y"][k], g["fs_h"][k], g["fs_guess"][k]) for k in range(n)])
    assert np.array_equal(got, g["fs_root"]), f"{(got != g['fs_root']).sum()} of {n} roots differ"


def test_danger_zone_counts(golden, oracle):
    g = golden("danger_golden.npz")
    S, fuel, cnt = g["dz_states"], g["dz_fuel"], g["dz_count"]
    got = np.array([oracle.danger_zone(S[k, 0:3], S[k, 3:6], S[k, 6:9], S[k, 9:12], fuel[k]) for k in range(len(S))])
    assert np.array_equal(got, cnt), f"{(got != cnt).sum()} of {len(cnt)} counts differ"


# ------------------------------------------------------------------ env (environment.py:66-255)
def test_cw_matrix_matches_reference(golden, oracle):
    g = golden("env_golden.npz")
    assert np.array_equal(oracle.cw_matrix(100.0), g["stm100_columns"])


@pytest.mark.parametrize("scen", ["cfg1", "long", "capt", "flag1"])
def test_env_rollout_bit_identical(golden, oracle, scen):
    g = {**golden("env_golden.npz"), **golden("env_capt_golden.npz")}
    env = oracle.Env(d_capture=float(g[f"{scen}_d_capture"]), max_episode_steps=int(g[f"{scen}_max_episode_steps"]),
                     M=g["stm100_columns"])
    flag = int(g[f"{scen}_flag"])
    s = env.reset(flag)
    assert np.array_equal(s, g[f"{scen}_reset_obs"])
    cnt = 0
    for t in range(len(g[f"{scen}_reward"])):
        cnt += 1
        obs, r, d = env.step(g[f"{scen}_pa"][t], g[f"{scen}_ea"][t], cnt)
        assert cnt == g[f"{scen}_count"][t]
        assert np.array_equal(obs, g[f"{scen}_obs"][t]), (scen, t)
        assert r == g[f"{scen}_reward"][t], (scen, t, r, g[f"{scen}_reward"][t])
        assert d == bool(g[f"{scen}_done"][t])
        assert env.e.dangerous_zone == g[f"{scen}_dz"][t]
        assert env.e.fuel_c == g[f"{scen}_fuel_c"][t] and env.e.fuel_t == g[f"{scen}_fuel_t"][t]
        assert env.e.dis == g[f"{scen}_dis"][t]
        if d:
            env.reset(flag)
            cnt = 0
    assert env.e.err == 0


# ------------------------------------------------------------------ normalisation (normalization.py)
def test_normalization_sequence(golden, oracle):
    g = golden("norm_golden.npz")
    rms = oracle.RunningMeanStd(18)
    for k in range(len(g["x"])):
        rms.update(g["x"][k])
        out = (g["x"][k] - rms.mean) / (rms.std + 1e-8)
        assert np.array_equal(out, g["x_normed"][k])
    assert rms.n == int(g["final_n"])
    assert np.array_equal(rms.mean, g["final_mean"]) and np.array_equal(rms.S, g["final_S"])


def test_chan_merge_equals_welford(golden, oracle):
    g = golden("norm_golden.npz")
    X = g["x"]
    n, mean, S = 0, np.zeros(18), np.zeros(18)
    for lo in range(0, len(X), 50):
        n, mean, S = oracle.chan_merge(n, mean, S, X[lo:lo + 50])
    np.testing.assert_allclose(mean, g["final_mean"], rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(S, g["final_S"], rtol=1e-10, atol=1e-6)


def test_reward_scaling_sequence(golden, oracle):
    g = golden("norm_golden.npz")
    rms = oracle.RunningMeanStd(1)
    R = np.zeros(1)
    for k in range(len(g["reward"])):
        R = 0.99 * R + g["reward"][k]
        rms.update(R)
        out = g["reward"][k] / (rms.std + 1e-8)
        assert float(np.ravel(out)[0]) == g["reward_scaled"][k]
        if g["done"][k]:
            R = np.zeros(1)


# ------------------------------------------------------------------ GAE / actor (ppo_continuous.py)
def test_gae_matches_reference_block(golden, oracle):
    g = golden("ppo_golden.npz")
    adv, vt = oracle.gae(g["gae_r"], g["gae_vs"], g["gae_vs_next"], g["gae_done"], g["gae_done"])
    # the reference recursion runs in fp32 under numpy 2 (SURVEY H4): the restatement is bit-identical
    assert np.array_equal(adv, g["gae_adv"])
    assert np.array_equal(vt, g["gae_v_target"])
    np.testing.assert_allclose(oracle.adv_normalize(adv), g["gae_adv_normed"], rtol=2e-6, atol=2e-6)


def test_actor_critic_forward(golden, oracle):
    g = golden("ppo_golden.npz")
    Wa = {k[len("actor."):]: g[k] for k in g.files if k.startswith("actor.")}
    Wc = {k[len("critic."):]: g[k] for k in g.files if k.startswith("critic.")}
    mean = oracle.actor_forward(Wa, g["obs"])
    # rows [0,384): raw env-scale observations (|x| ~ 1e5, pre-activations ~1e5 in fp32); rows [384,768): unit scale
    np.testing.assert_allclose(mean[:384], g["mean"][:384], rtol=0, atol=1e-4)
    np.testing.assert_allclose(mean[384:], g["mean"][384:], rtol=0, atol=5e-6)
    a, lp = oracle.gaussian_sample(g["mean"], Wa["log_std"], g["eps"])
    np.testing.assert_allclose(a, g["action"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(lp, g["logp"], rtol=1e-5, atol=1e-5)
    v = oracle.critic_forward(Wc, g["obs"])
    np.testing.assert_allclose(v, g["value"], rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------ Numerical_calculation_method (scipy RK45 on the CW ODE)
def test_cw_ode_rk45_matches_reference(golden, oracle):
    g = golden("ode_golden.npz")
    for k in range(len(g["t"])):
        for y0, ref in ((g["state_c"][k], g["out_c"][k]), (g["state_t"][k], g["out_t"][k])):
            y, nsteps = oracle.cw_ode_rk45(y0, g["t"][k])
            assert 2 <= nsteps <= 8
            np.testing.assert_allclose(y, ref, rtol=2e-12, atol=1e-9)


# ------------------------------------------------------------------ reachable-domain sweep (RD_single_pulse.py:40-148)
def test_reachable_domain_sweep_matches_reference(golden, oracle):
    g = golden("reach_golden.npz")
    N = int(g["N"])
    for n in range(len(g["idx"])):
        hi, lo, valid = oracle.reachable_domain(g["elements"][n], g["delta_max"][n], N, N)
        assert hi.shape == g[f"rf_max_{n}"].shape and valid.sum() > 10
        np.testing.assert_allclose(hi, g[f"rf_max_{n}"], rtol=1e-12, atol=1e-6)
        np.testing.assert_allclose(lo, g[f"rf_min_{n}"], rtol=1e-12, atol=1e-6)


def test_env_flag2_dynamics_match_reference(golden, oracle):
    """Flag 2 (environment.py:257-316; the two surrogate-fit calls stubbed when the fixture was recorded): 80 Flag-0 steps,
    then reset(2) and 500 Flag-2 steps, bit for bit (obs, reward, done, persistent dz / fuel / dis)."""
    g = golden("env_flag2_golden.npz")
    eg = golden("env_golden.npz")
    env = oracle.Env(d_capture=float(g["d_capture"]), d_range=float(g["d_range"]), max_episode_steps=int(g["max_episode_steps"]),
                     M=eg["stm100_columns"])
    env.reset(0)
    for t in range(len(g["flag"])):
        if t > 0 and g["flag"][t] != g["flag"][t - 1]:
            env.reset(int(g["flag"][t]))
        o, r, d = env.step(g["pa"][t], g["ea"][t], int(g["count"][t]))
        assert np.array_equal(o, g["obs"][t]) and r == g["reward"][t] and d == bool(g["done"][t]), t
        assert env.e.dangerous_zone == g["dz"][t] and env.e.fuel_c == g["fuel_c"][t] and env.e.dis == g["dis"][t], t
        if d:
            env.reset(int(g["flag"][t]))
    assert (g["flag"] == 2).sum() == 500 and g["done"][80:].sum() >= 5
