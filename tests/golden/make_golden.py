"""Generates the committed golden fixtures by RUNNING THE REFERENCE ITSELF in the build container.

    python tests/golden/make_golden.py            # needs /root/reference (read-only)

Container used for the committed files: Python 3.12.3, numpy 2.3.5 (scipy-openblas 0.3.30 Haswell
kernels), scipy 1.18.1, torch 2.11.0 CPU, glibc libm, Intel Xeon (AVX-512). The GPU box has no
reference tree: tests there read only the .npz files written here.

Each fixture stores inputs and the reference's outputs; nothing here comes from the oracle or
from the CUDA path.
"""
from __future__ import annotations

import contextlib
import io
import os
import re
import sys
import textwrap
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import refshim  # noqa: E402

warnings.filterwarnings("ignore")
REF = refshim.REF


def save(name, **arrs):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrs)
    print(f"wrote {name}: " + ", ".join(f"{k}{tuple(np.shape(v))}" for k, v in arrs.items()),
          f"[{os.path.getsize(path) / 1024:.0f} KiB]")


# --------------------------------------------------------------------------------------------
def config2_orbits(n=4096, seed=0):
    """SURVEY.md 8(d) config 2: rows [0, n/2) LEO, [n/2, n) GEO; states via the reference's
    calculate_state_information (km, km/s)."""
    sf = refshim.load()["satellite_function"]
    rng = np.random.default_rng(seed)
    h = n // 2
    a = np.concatenate([rng.uniform(6778, 7378, h), 42164 + rng.uniform(-50, 50, n - h)])
    e = np.concatenate([rng.uniform(1e-4, 0.02, h), rng.uniform(1e-4, 0.005, n - h)])
    inc = np.concatenate([rng.uniform(0.01, np.pi - 0.01, h), rng.uniform(1e-3, 0.1, n - h)])
    om, Om, f = (rng.uniform(0, 2 * np.pi, n) for _ in range(3))
    el = np.stack([a, e, inc, om, Om, f], axis=1)
    X = np.empty((6, n))
    for k in range(n):
        R, V = sf.Time_window_of_danger_zone.calculate_state_information(list(el[k]), miu=398600)
        X[:3, k], X[3:, k] = R, V
    return el, X


def gen_rk4():
    el, X0 = config2_orbits()
    out = {"elements": el, "x0": X0}
    for tag, j2 in (("j2off", 0.0), ("j2on", None)):
        ns = refshim.load_rk4_script(j2)
        RK = ns["RungeKutta"]
        x = X0.copy()
        for i in range(1000):
            x = RK(i * 1.0, x, 1.0)
        out[f"x1000_{tag}"] = x
        # scalar path (as shipped: one state per call) on 8 orbits, to show batched == scalar
        idx = np.array([0, 1, 2, 3, 2048, 2049, 2050, 4095])
        xs = X0[:, idx].copy()
        for c in range(len(idx)):
            rv = xs[:, c].copy()
            for i in range(1000):
                rv = RK(i * 1.0, rv, 1.0)
            xs[:, c] = rv
        out[f"scalar_idx"] = idx
        out[f"x1000_scalar_{tag}"] = xs
    # the script's own initial condition (:46), 86 400 steps of 1 s (what `print(RV0)` at :52 emits)
    ns = refshim.load_rk4_script(None)
    rv = np.array([3971.676026, -2202.172866, -5161.178823, 6.059801, 3.231769, 3.293050])
    out["script_ic"] = rv.copy()
    for i in range(86400):
        rv = ns["RungeKutta"](i * 1, rv, 1)
    out["script_86400"] = rv
    # a few StateEq evaluations
    pts = X0[:, ::512].T.copy()
    out["stateeq_in"] = pts
    out["stateeq_out"] = np.array([ns["StateEq"](0, p) for p in pts])
    save("rk4_golden.npz", **out)


# --------------------------------------------------------------------------------------------
def gen_elements():
    """The reference's only known-answer data: spacecraft_state.txt <-> all_input.csv (841 rows)."""
    sf = refshim.load()["satellite_function"]
    txt = open(os.path.join(REF, "single_pluse_model", "spacecraft_state.txt"), encoding="utf-8-sig").read()
    txt = txt.replace("\n", " ")
    recs = re.findall(r"R0_c, V0_c, fuel_c: \[([^\]]*)\] \[([^\]]*)\] ([-0-9.e+]+)", txt)
    R = np.array([[float(t) for t in r[0].split()] for r in recs])
    V = np.array([[float(t) for t in r[1].split()] for r in recs])
    fuel = np.array([float(r[2]) for r in recs])
    csv = np.genfromtxt(os.path.join(REF, "single_pluse_model", "all_input.csv"), delimiter=",", skip_header=1)
    if csv.shape[0] != len(recs):  # no header row
        csv = np.genfromtxt(os.path.join(REF, "single_pluse_model", "all_input.csv"), delimiter=",")
    assert csv.shape[0] == len(recs) == 841, (csv.shape, len(recs))
    # full six elements from the live reference for the same states (the csv holds a,e,i,f,fuel only)
    full = np.array([sf.Time_window_of_danger_zone.calculate_orbital_elements(3.986e14, R[k], V[k])
                     for k in range(len(recs))])
    # round trip through calculate_state_information
    rt = np.array([np.concatenate(sf.Time_window_of_danger_zone.calculate_state_information(list(full[k]), miu=3.986e14))
                   for k in range(len(recs))])
    save("elements_golden.npz", R=R, V=V, fuel=fuel, csv_a_e_i_f_fuel=csv, elements_live=full, state_roundtrip=rt)


# --------------------------------------------------------------------------------------------
def run_env(flag, d_capture, max_steps, n_steps, seed, action_scale=2.0):
    """drives the reference env exactly like CPPO_main.py:111-153 does (reset on done)."""
    env = refshim.make_env(d_capture, max_steps)
    rng = np.random.default_rng(seed)
    acts_p = rng.uniform(-action_scale, action_scale, (n_steps, 3)).astype(np.float32).astype(np.float64)
    acts_e = rng.uniform(-action_scale, action_scale, (n_steps, 3)).astype(np.float32).astype(np.float64)
    # sprinkle exact zeros / exact limits so pv4's zero test and the clip are exercised
    zero_rows = rng.choice(n_steps, n_steps // 25, replace=False)
    acts_p[zero_rows, rng.integers(0, 3, len(zero_rows))] = 0.0
    obs0 = []
    obs, rew, done, dz, fuel_c, fuel_t, dis, cnts = [], [], [], [], [], [], [], []
    s = env.reset(flag)
    obs0.append(np.asarray(s, dtype=np.float64))
    cnt = 0
    for t in range(n_steps):
        cnt += 1
        s_, r, d = refshim.quiet_step(env, acts_p[t], acts_e[t], cnt)
        obs.append(np.asarray(s_, dtype=np.float64)); rew.append(float(r)); done.append(bool(d))
        dz.append(int(env.dangerous_zone)); fuel_c.append(float(env.fuel_c)); fuel_t.append(float(env.fuel_t))
        dis.append(float(env.dis)); cnts.append(cnt)
        if d:
            s = env.reset(flag)
            cnt = 0
    return dict(pa=acts_p, ea=acts_e, obs=np.array(obs), reward=np.array(rew), done=np.array(done),
                dz=np.array(dz, dtype=np.int32), fuel_c=np.array(fuel_c), fuel_t=np.array(fuel_t),
                dis=np.array(dis), count=np.array(cnts, dtype=np.int32), reset_obs=obs0[0],
                d_capture=np.float64(d_capture), max_episode_steps=np.int32(max_steps), flag=np.int32(flag))


def gen_env():
    mods = refshim.load()
    cw = mods["satellite_function"].Clohessy_Wiltshire(np.zeros(3), np.zeros(3), np.zeros(3), np.zeros(3))
    # the STM the reference uses (matrix = identity applied column by column through its own code)
    M = np.array([cw.__class__(np.eye(6)[k, :3], np.eye(6)[k, 3:], np.zeros(3), np.zeros(3)).State_transition_matrix(100)[0]
                  for k in range(6)]).T
    out = {"stm100_columns": M}
    scen = {
        "cfg1": dict(flag=0, d_capture=20000, max_steps=64, n_steps=640, seed=11),     # config 1 plumbing shape
        "long": dict(flag=0, d_capture=20000, max_steps=1000, n_steps=3000, seed=1),   # config 3 parity shape
        "capt": dict(flag=0, d_capture=181000, max_steps=200, n_steps=1500, seed=5),   # capture branch
        "flag1": dict(flag=1, d_capture=181500, max_steps=150, n_steps=1200, seed=7),  # evader training branch
    }
    for name, kw in scen.items():
        res = run_env(**kw)
        for k, v in res.items():
            out[f"{name}_{k}"] = v
        print(name, "episodes:", int(res["done"].sum()), "dz hist:", np.bincount(res["dz"], minlength=3),
              "captures:", int(((res["reward"] == 100) & res["done"]).sum()))
    # the capture scenario gets a file of its own so that each fixture stays under 1 MB
    save("env_golden.npz", **{k: v for k, v in out.items() if not k.startswith("capt_")})
    save("env_capt_golden.npz", **{k: v for k, v in out.items() if k.startswith("capt_")})


def gen_env_flag2():
    """Flag 2 (environment.py:257-316): the reference's own step with the two surrogate calls (:299 numerical_method_process,
    :301 trian_elliptical_fitting.train - the reachable-domain network fit, outside the hot path) replaced by no-ops.
    Phase A = 80 Flag-0 steps from reset(0), so that fuel / dis / dangerous_zone (which persist through reset, Q2, and gate the
    Flag-2 impulse) are non-trivial; phase B = reset(2) and 500 Flag-2 steps with resets on done."""
    mods = refshim.load()
    mods["environment"].real_time_data_process.numerical_method_process = lambda *a, **k: None
    env = refshim.make_env(d_capture=181200, max_episode_steps=60)
    env.trian_elliptical_fitting.train = lambda *a, **k: None
    env.d_range = 250000.0          # > the 182 km starting distance: the "pursuer frozen" gating branch (:265-270) is exercised
    rng = np.random.default_rng(29)
    nA, nB = 80, 500
    n = nA + nB
    pa = rng.uniform(-2, 2, (n, 3)).astype(np.float32).astype(np.float64)
    ea = rng.uniform(-2, 2, (n, 3)).astype(np.float32).astype(np.float64)
    flags = np.array([0] * nA + [2] * nB, dtype=np.int32)
    obs, rew, done, dz, fuel_c, fuel_t, dis, cnts = [], [], [], [], [], [], [], []
    env.reset(0)
    cnt = 0
    for t in range(n):
        if t == nA:
            env.reset(2); cnt = 0
        cnt += 1
        s_, r, d = refshim.quiet_step(env, pa[t], ea[t], cnt)
        obs.append(np.asarray(s_, dtype=np.float64)); rew.append(float(r)); done.append(bool(d))
        dz.append(int(env.dangerous_zone)); fuel_c.append(float(env.fuel_c)); fuel_t.append(float(env.fuel_t))
        dis.append(float(env.dis)); cnts.append(cnt)
        if d:
            env.reset(int(flags[t])); cnt = 0
    save("env_flag2_golden.npz", pa=pa, ea=ea, flag=flags, obs=np.array(obs), reward=np.array(rew), done=np.array(done),
         dz=np.array(dz, dtype=np.int32), fuel_c=np.array(fuel_c), fuel_t=np.array(fuel_t), dis=np.array(dis),
         count=np.array(cnts, dtype=np.int32), d_capture=np.float64(181200), d_range=np.float64(250000),
         max_episode_steps=np.int32(60))
    print("flag2: episodes", int(np.sum(done[nA:])), "frozen-pursuer steps", int(np.sum((np.array(dz[nA - 1:-1]) != 0))), "dz hist", np.bincount(dz, minlength=3))


# --------------------------------------------------------------------------------------------
def gen_fsolve_dz():
    sf = refshim.load()["satellite_function"]
    rng = np.random.default_rng(3)
    # (a) raw Numerical_iteration_method cases
    obj = sf.Time_window_of_danger_zone(R0_c=np.array([27298000.0, 32306000.0, 0.0]), V0_c=np.array([-2350.0, 1970.0, 0.1]),
                                        R0_t=np.array([27116000.0, 32306000.0, 10.0]), V0_t=np.array([-2350.0, 1970.0, 0.2]),
                                        Delta_V_c=300.0, time_step=1)
    n = 4000
    dvm = 10 ** rng.uniform(-1, 3.5, n)
    theta = np.where(rng.random(n) < 0.1, 0.0, rng.uniform(0, 2 * np.pi, n))
    v1x = rng.normal(0, 30, n)
    v1y = 3074 + rng.normal(0, 50, n) + dvm * rng.choice([-1, 1], n)
    h = 4.2164e7 * v1y * (1 + rng.normal(0, 1e-3, n))
    guess = rng.choice([np.pi / 2, -np.pi / 2], n)
    root = np.array([obj.Numerical_iteration_method(dvm[k], theta[k], v1x[k], v1y[k], h[k], guess[k]) for k in range(n)])
    # (b) danger-zone counts on states visited by the env + random perturbations of them
    env = refshim.make_env(20000, 400)
    states, fuels, counts = [], [], []
    s = env.reset(0)
    cnt = 0
    Rcw, Vcw = np.array([27098000.0, 32306000.0, 0.0]), np.array([-2350.0, 1970.0, 0.0])
    for t in range(1500):
        cnt += 1
        pa = rng.uniform(-2, 2, 3).astype(np.float32).astype(np.float64)
        ea = rng.uniform(-2, 2, 3).astype(np.float32).astype(np.float64)
        s_, r, d = refshim.quiet_step(env, pa, ea, cnt)
        if not d:
            P, Pv, E, Ev = s_[6:9], s_[9:12], s_[12:15], s_[15:18]
            states.append(np.concatenate([Rcw + P, Vcw + Pv, Rcw + E, Vcw + Ev]))
            fuels.append(float(env.fuel_c)); counts.append(int(env.dangerous_zone))
        else:
            env.reset(0); cnt = 0
    states = np.array(states); fuels = np.array(fuels); counts = np.array(counts, dtype=np.int32)
    # random perturbed states with a wider spread of fuel / geometry
    m = 1500
    base = states[rng.integers(0, len(states), m)].copy()
    base[:, 0:3] += rng.normal(0, 5e4, (m, 3)); base[:, 6:9] += rng.normal(0, 5e4, (m, 3))
    base[:, 3:6] += rng.normal(0, 20, (m, 3)); base[:, 9:12] += rng.normal(0, 20, (m, 3))
    fuel2 = rng.uniform(-600, 320, m)
    cnt2 = []
    with contextlib.redirect_stdout(io.StringIO()):
        for k in range(m):
            o = sf.Time_window_of_danger_zone(R0_c=base[k, 0:3].copy(), V0_c=base[k, 3:6].copy(), R0_t=base[k, 6:9].copy(),
                                              V0_t=base[k, 9:12].copy(), Delta_V_c=fuel2[k], time_step=1)
            cnt2.append(o.calculate_number_of_hanger_area())
    save("danger_golden.npz", fs_dvm=dvm, fs_theta=theta, fs_v1x=v1x, fs_v1y=v1y, fs_h=h, fs_guess=guess, fs_root=root,
         dz_states=np.concatenate([states, base]), dz_fuel=np.concatenate([fuels, fuel2]),
         dz_count=np.concatenate([counts, np.array(cnt2, dtype=np.int32)]))
    print("dz hist", np.bincount(np.concatenate([counts, cnt2]), minlength=3))


# --------------------------------------------------------------------------------------------
def gen_ppo():
    import torch
    mods = refshim.load()
    ppo = mods["ppo_continuous"]
    args = refshim.Args(policy_dist="Gaussian", max_action=1.6, batch_size=2048, mini_batch_size=64,
                        max_train_steps=5000, lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1,
                        K_epochs=10, entropy_coef=0.01, set_adam_eps=True, use_grad_clip=True, use_lr_decay=True,
                        use_adv_norm=True, state_dim=18, action_dim=3, hidden_width=256, use_tanh=True,
                        use_orthogonal_init=True, chkpt_dir=os.path.join(REF, "model_file", "one_layer"))
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        agent = ppo.PPO_continuous(args, "pursuer")
    agent.load_checkpoint()  # the only shipped pair whose shapes match (SURVEY.md s4)
    rng = np.random.default_rng(9)
    out = {}
    for k, v in agent.actor.state_dict().items():
        out["actor." + k] = v.numpy().copy()
    for k, v in agent.critic.state_dict().items():
        out["critic." + k] = v.numpy().copy()
    # observations: env-like magnitudes (raw, unnormalised as the shipped driver feeds them) and unit-scale ones
    env_g = np.load(os.path.join(HERE, "env_golden.npz"))
    obs_env = env_g["long_obs"][:384].astype(np.float32)
    obs_unit = rng.normal(0, 1, (384, 18)).astype(np.float32)
    obs = np.concatenate([obs_env, obs_unit])
    with torch.no_grad():
        s = torch.tensor(obs)
        mean = agent.actor(s)
        dist = agent.actor.get_dist(s)
        eps = torch.tensor(rng.normal(0, 1, (obs.shape[0], 3)).astype(np.float32))
        std = torch.exp(agent.actor.log_std.expand_as(mean))
        a = torch.clamp(mean + std * eps, -1.6, 1.6)   # == dist.sample() with the normal draw made explicit (H6)
        logp = dist.log_prob(a)
        v = agent.critic(s)
    out.update(obs=obs, mean=mean.numpy(), eps=eps.numpy(), action=a.numpy(), logp=logp.numpy(), value=v.numpy().ravel())

    # GAE: execute the reference's own lines 198-210 of ppo_continuous.py on a synthetic buffer
    src = open(os.path.join(REF, "ppo_continuous.py"), encoding="utf-8").read().splitlines()
    block = textwrap.dedent("\n".join(src[197:210]))
    B = 2048
    r = rng.normal(0, 2, (B, 1)).astype(np.float32)
    done = (rng.random((B, 1)) < 0.02).astype(np.float32)
    r[done[:, 0] > 0] = 100.0
    sB = torch.tensor(rng.normal(0, 1, (B, 18)).astype(np.float32))
    s_B = torch.cat([sB[1:], torch.tensor(rng.normal(0, 1, (1, 18)).astype(np.float32))])

    class _Self:
        pass
    me = _Self()
    me.critic, me.gamma, me.lamda, me.use_adv_norm = agent.critic, 0.99, 0.95, True
    ns = dict(self=me, torch=torch, s=sB, s_=s_B, r=torch.tensor(r), dw=torch.tensor(done), done=torch.tensor(done))
    exec(block, ns)
    with torch.no_grad():
        vs, vs_ = agent.critic(sB), agent.critic(s_B)
    out.update(gae_r=r.ravel(), gae_done=done.ravel(), gae_vs=vs.numpy().ravel(), gae_vs_next=vs_.numpy().ravel(),
               gae_adv_normed=ns["adv"].numpy().ravel(), gae_v_target=ns["v_target"].numpy().ravel())
    # un-normalised advantages: same block with use_adv_norm False
    me.use_adv_norm = False
    ns = dict(self=me, torch=torch, s=sB, s_=s_B, r=torch.tensor(r), dw=torch.tensor(done), done=torch.tensor(done))
    exec(block, ns)
    out.update(gae_adv=ns["adv"].numpy().ravel())
    save("ppo_golden.npz", **out)


# --------------------------------------------------------------------------------------------
def gen_norm():
    norm = refshim.load()["normalization"]
    env_g = np.load(os.path.join(HERE, "env_golden.npz"))
    X = env_g["long_obs"][:300]
    rew = env_g["long_reward"][:300]
    done = env_g["long_done"][:300]
    nz = norm.Normalization(shape=18)
    xn = np.array([nz(X[k].copy()) for k in range(len(X))])
    mean_hist = None
    rs = norm.RewardScaling(shape=1, gamma=0.99)
    rsc = []
    for k in range(len(rew)):
        rsc.append(float(np.ravel(rs(rew[k]))[0]))
        if done[k]:
            rs.reset()
    save("norm_golden.npz", x=X, x_normed=xn, final_mean=np.asarray(nz.running_ms.mean, dtype=np.float64),
         final_S=np.asarray(nz.running_ms.S, dtype=np.float64), final_std=np.asarray(nz.running_ms.std, dtype=np.float64),
         final_n=np.int64(nz.running_ms.n), reward=rew, done=done, reward_scaled=np.array(rsc),
         rs_final_std=np.asarray(rs.running_ms.std, dtype=np.float64))


def gen_ode():
    """Numerical_calculation_method.numerical_calculation (scipy RK45 on the CW ODE), satellite_function.py:783-839"""
    sf = refshim.load()["satellite_function"]
    rng = np.random.default_rng(21)
    n = 240
    sc = np.where((np.arange(n) % 2 == 0)[:, None], np.concatenate([rng.normal(0, 2e5, (n, 3)), rng.normal(0, 3, (n, 3))], axis=1),
                  np.concatenate([rng.normal(0, 100, (n, 3)), rng.normal(0, 0.01, (n, 3))], axis=1))
    st = np.concatenate([rng.normal(0, 5e4, (n, 3)), rng.normal(0, 2, (n, 3))], axis=1)
    ts = np.array([100, 600, 50, 1000] * (n // 4), dtype=np.float64)
    oc, ot = [], []
    for k in range(n):
        a, b = sf.Numerical_calculation_method(R0_c=sc[k, :3].copy(), V0_c=sc[k, 3:].copy(), R0_t=st[k, :3].copy(),
                                               V0_t=st[k, 3:].copy()).numerical_calculation(int(ts[k]))
        oc.append(a); ot.append(b)
    save("ode_golden.npz", state_c=sc, state_t=st, t=ts, out_c=np.array(oc), out_t=np.array(ot))


def gen_reach():
    """RD_single_pulse.Reachable_Domain point clouds (captured before the ellipse fit), reduced sweep N2 = N3 = 40"""
    import importlib
    refshim.load()
    sys.path.insert(0, REF)
    RD = importlib.import_module("single_pluse_model.RD_single_pulse")
    cap = {}
    RD.cf.Curve_fitting = lambda a, b: (cap.__setitem__("a", a), cap.__setitem__("b", b), [0] * 10)[2]
    RD.params["N2"], RD.params["N3"] = 40, 40
    g = np.load(os.path.join(HERE, "elements_golden.npz"))
    idx = np.array([0, 100, 300, 500, 700, 840])
    out = {"idx": idx, "elements": g["elements_live"][idx], "delta_max": g["fuel"][idx], "N": np.int32(40)}
    for n, k in enumerate(idx):
        RD.Incoming_parameters(list(g["elements_live"][k]), float(g["fuel"][k]))
        out[f"rf_max_{n}"], out[f"rf_min_{n}"] = np.asarray(cap["a"]), np.asarray(cap["b"])
    save("reach_golden.npz", **out)


if __name__ == "__main__":
    which = sys.argv[1:] or ["rk4", "elements", "env", "flag2", "danger", "ppo", "norm", "ode", "reach"]
    if "rk4" in which: gen_rk4()
    if "elements" in which: gen_elements()
    if "env" in which: gen_env()
    if "flag2" in which: gen_env_flag2()
    if "danger" in which: gen_fsolve_dz()
    if "ppo" in which: gen_ppo()
    if "norm" in which: gen_norm()
    if "ode" in which: gen_ode()
    if "reach" in which: gen_reach()
