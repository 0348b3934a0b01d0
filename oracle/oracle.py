"""ctypes binding of the CPU oracle (oracle/sat_oracle.c).

TEST INFRASTRUCTURE ONLY. Allowed importers: tests/, __graft_entry__.smoke(), and bench.py's
cpu_baseline / --impl reference legs. The product package (ppo-rl-satellite_b200/) must never
import this module; tests/test_cabi_symbols.py::test_product_never_imports_the_oracle enforces that.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libsat_oracle.so")

# constants of the reference (script :9-11, environment.py:338-339, satellite_function.py:28)
MU_KM, RE_KM, J2 = 398600.0, 6378.137, 0.00108263
MU_M, RE_M = 3.986e14, 6378137.0
R_CW = np.array([27098000.0, 32306000.0, 0.0])
V_CW = np.array([-2350.0, 1970.0, 0.0])


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "sat_oracle.c")
    hdr = os.path.join(_HERE, "sat_oracle.h")
    if (not force and os.path.exists(_SO)
            and os.path.getmtime(_SO) >= max(os.path.getmtime(src), os.path.getmtime(hdr))):
        return _SO
    subprocess.run(["make", "-C", _HERE, "-s", "-B"], check=True)
    return _SO


class OrcEnv(C.Structure):
    _fields_ = [("P", C.c_double * 3), ("Pv", C.c_double * 3), ("E", C.c_double * 3), ("Ev", C.c_double * 3),
                ("fuel_c", C.c_double), ("fuel_t", C.c_double), ("dis", C.c_double),
                ("dangerous_zone", C.c_int32), ("int_state", C.c_int32), ("flag", C.c_int32), ("err", C.c_int32),
                ("d_capture", C.c_double), ("d_range", C.c_double), ("max_episode_steps", C.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        L = _lib
        dp, fp, i64, i32 = C.POINTER(C.c_double), C.POINTER(C.c_float), C.c_int64, C.c_int
        L.orc_rk4_batch.argtypes = [dp, i64, i64, C.c_double, i32, C.c_double, C.c_double, C.c_double, i32]
        L.orc_rk4_step.argtypes = [dp, C.c_double, C.c_double, C.c_double, C.c_double]
        L.orc_state_eq.argtypes = [dp, C.c_double, C.c_double, C.c_double, dp]
        L.orc_cw_matrix.argtypes = [C.c_double, dp]
        L.orc_cw_apply.argtypes = [dp, dp, dp]
        L.orc_orbital_elements.argtypes = [C.c_double, dp, dp, dp]
        L.orc_orbital_elements.restype = i32
        L.orc_state_information.argtypes = [dp, C.c_double, dp, dp]
        L.orc_numerical_iteration.argtypes = [C.c_double] * 7
        L.orc_numerical_iteration.restype = C.c_double
        L.orc_danger_zone.argtypes = [dp, dp, dp, dp, C.c_double, C.c_double]
        L.orc_danger_zone.restype = i32
        L.orc_danger_zone_debug.argtypes = [dp, dp, dp, dp, C.c_double, C.c_double, dp]
        L.orc_danger_zone_debug.restype = i32
        L.orc_cw_ode_rk45.argtypes = [dp, C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_int)]
        L.orc_cw_ode_rk45.restype = i32
        L.orc_reachable_domain.argtypes = [dp, C.c_double, i32, i32, C.c_double, dp, dp, C.POINTER(C.c_uint8)]
        L.orc_env_init.argtypes = [C.POINTER(OrcEnv), C.c_double, C.c_double, C.c_double, C.c_double, i32]
        L.orc_env_reset.argtypes = [C.POINTER(OrcEnv), i32, dp]
        L.orc_env_step.argtypes = [C.POINTER(OrcEnv), dp, dp, dp, i32, dp, dp]
        L.orc_env_step.restype = i32
        L.orc_env_step_rk4.argtypes = [C.POINTER(OrcEnv), C.c_double, i32, C.c_double, C.c_double, C.c_double,
                                       dp, dp, i32, dp, dp]
        L.orc_env_step_rk4.restype = i32
        L.orc_env_last_terms.argtypes = [dp]
        L.orc_env_step_batch.argtypes = [C.POINTER(OrcEnv), C.POINTER(C.c_int32), i64, dp, dp, dp, dp, dp,
                                         C.POINTER(C.c_uint8), i32, i32]
        L.orc_env_step_rk4_batch.argtypes = [C.POINTER(OrcEnv), C.POINTER(C.c_int32), i64, C.c_double, i32,
                                             C.c_double, C.c_double, C.c_double, dp, dp, dp, dp,
                                             C.POINTER(C.c_uint8), i32, i32]
        L.orc_gae.argtypes = [fp, fp, fp, fp, fp, i64, C.c_double, C.c_double, fp, fp]
        L.orc_adv_normalize.argtypes = [fp, i64]
        L.orc_actor_forward.argtypes = [fp] * 6 + [i32, i32, i32, C.c_float, fp, i64, fp]
        L.orc_critic_forward.argtypes = [fp] * 6 + [i32, i32, fp, i64, fp]
        L.orc_gaussian_sample.argtypes = [fp, fp, fp, i64, i32, C.c_float, fp, fp]
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


# ------------------------------------------------------------------ RK4
def rk4_propagate(x, h, steps, mu=MU_KM, re=RE_KM, j2=J2, nthreads=1):
    """x: (6, N) float64 -> new (6, N) after `steps` RungeKutta calls (script :34-40)."""
    x = _f64(x).copy()
    n = x.shape[1]
    lib().orc_rk4_batch(_dp(x), n, n, float(h), int(steps), mu, re, j2, int(nthreads))
    return x


def state_eq(rv, mu=MU_KM, re=RE_KM, j2=J2):
    rv = _f64(rv)
    f = np.empty(6)
    lib().orc_state_eq(_dp(rv), mu, re, j2, _dp(f))
    return f


# ------------------------------------------------------------------ CW
def cw_matrix(t=100.0):
    M = np.empty(36)
    lib().orc_cw_matrix(float(t), _dp(M))
    return M.reshape(6, 6)


def cw_apply(M, s):
    M = _f64(M).ravel()
    s = _f64(s)
    out = np.empty(6)
    lib().orc_cw_apply(_dp(M), _dp(s), _dp(out))
    return out


def cw_ode_constants():
    """(2*omega, 3*omega**2, omega**2) exactly as orbit_ode computes them (satellite_function.py:796-801, 818-820)"""
    import math
    mu, r = 398600, 35786
    omega = math.sqrt(mu / (r ** 3))
    return 2 * omega, 3 * omega ** 2, omega ** 2


def cw_ode_rk45(y0, t):
    y = _f64(y0).copy()
    w2, w3, wz = cw_ode_constants()
    ns = C.c_int()
    rc = lib().orc_cw_ode_rk45(_dp(y), float(t), w2, w3, wz, C.byref(ns))
    assert rc == 0
    return y, ns.value


# ------------------------------------------------------------------ elements / danger zone
def orbital_elements(miu, R0, V0):
    R0, V0 = _f64(R0), _f64(V0)
    out = np.zeros(6)
    k = lib().orc_orbital_elements(float(miu), _dp(R0), _dp(V0), _dp(out))
    return out[:k]


def state_information(el, miu=MU_M):
    el = _f64(el)
    R, V = np.empty(3), np.empty(3)
    lib().orc_state_information(_dp(el), float(miu), _dp(R), _dp(V))
    return R, V


def numerical_iteration(u, dvm, theta, v1x, v1y, h, guess):
    return lib().orc_numerical_iteration(u, dvm, theta, v1x, v1y, h, guess)


def danger_zone(Rc, Vc, Rt, Vt, dv, u=MU_M):
    Rc, Vc, Rt, Vt = map(_f64, (Rc, Vc, Rt, Vt))
    return lib().orc_danger_zone(_dp(Rc), _dp(Vc), _dp(Rt), _dp(Vt), float(dv), float(u))


def danger_zone_debug(Rc, Vc, Rt, Vt, dv, u=MU_M):
    Rc, Vc, Rt, Vt = map(_f64, (Rc, Vc, Rt, Vt))
    dbg = np.zeros(16)
    c = lib().orc_danger_zone_debug(_dp(Rc), _dp(Vc), _dp(Rt), _dp(Vt), float(dv), float(u), _dp(dbg))
    return c, dbg.reshape(2, 8)


def reachable_domain(el, delta_max, N2=200, N3=200, u=MU_M):
    """RD_single_pulse.Reachable_Domain sweep -> (RF_max [K,3], RF_min [K,3]) in the reference's append order, plus the mask"""
    el = _f64(el)
    m = (N2 + 1) * (N3 + 1)
    hi, lo = np.zeros((m, 3)), np.zeros((m, 3))
    valid = np.zeros(m, dtype=np.uint8)
    lib().orc_reachable_domain(_dp(el), float(delta_max), int(N2), int(N3), float(u), _dp(hi), _dp(lo),
                               valid.ctypes.data_as(C.POINTER(C.c_uint8)))
    v = valid.astype(bool)
    return hi[v], lo[v], v


# ------------------------------------------------------------------ env
class Env:
    """Scalar env with the reference's reset/step contract (environment.py:66-179)."""

    def __init__(self, d_capture=100000.0, d_range=100000.0, fuel_c=320.0, fuel_t=320.0,
                 max_episode_steps=1000, M=None):
        self.e = OrcEnv()
        lib().orc_env_init(C.byref(self.e), d_capture, d_range, fuel_c, fuel_t, max_episode_steps)
        self.M = _f64(cw_matrix(100.0) if M is None else M).ravel().copy()

    def reset(self, flag=0):
        obs = np.empty(18)
        lib().orc_env_reset(C.byref(self.e), int(flag), _dp(obs))
        return obs

    def step(self, pa, ea, count):
        pa, ea = _f64(pa), _f64(ea)
        obs = np.empty(18)
        r = C.c_double()
        d = lib().orc_env_step(C.byref(self.e), _dp(self.M), _dp(pa), _dp(ea), int(count), _dp(obs), C.byref(r))
        return obs, r.value, bool(d)

    def step_rk4(self, pa, ea, count, h=1.0, substeps=100, mu=MU_M, re=RE_M, j2=J2):
        pa, ea = _f64(pa), _f64(ea)
        obs = np.empty(18)
        r = C.c_double()
        d = lib().orc_env_step_rk4(C.byref(self.e), h, substeps, mu, re, j2, _dp(pa), _dp(ea), int(count),
                                   _dp(obs), C.byref(r))
        return obs, r.value, bool(d)

    def last_terms(self):
        t = np.empty(7)
        lib().orc_env_last_terms(_dp(t))
        return t


class BatchEnv:
    """n independent scalar envs with per-env counters and auto-reset (the batched contract)."""

    def __init__(self, n, d_capture=100000.0, d_range=100000.0, fuel_c=320.0, fuel_t=320.0,
                 max_episode_steps=1000, flag=0, M=None, nthreads=1):
        self.n = n
        self.envs = (OrcEnv * n)()
        for i in range(n):
            lib().orc_env_init(C.byref(self.envs[i]), d_capture, d_range, fuel_c, fuel_t, max_episode_steps)
            lib().orc_env_reset(C.byref(self.envs[i]), flag, None)
        self.counts = np.zeros(n, dtype=np.int32)
        self.M = _f64(cw_matrix(100.0) if M is None else M).ravel().copy()
        self.nthreads = nthreads

    def set_state(self, P, Pv, E, Ev):
        for i in range(self.n):
            e = self.envs[i]
            for k in range(3):
                e.P[k], e.Pv[k], e.E[k], e.Ev[k] = P[i, k], Pv[i, k], E[i, k], Ev[i, k]
            e.int_state = 0

    def state(self):
        out = np.empty((self.n, 12))
        for i in range(self.n):
            e = self.envs[i]
            out[i] = list(e.P) + list(e.Pv) + list(e.E) + list(e.Ev)
        return out

    def aux(self):
        return (np.array([e.fuel_c for e in self.envs]), np.array([e.fuel_t for e in self.envs]),
                np.array([e.dis for e in self.envs]), np.array([e.dangerous_zone for e in self.envs]))

    def step(self, pa, ea, auto_reset=True):
        pa, ea = _f64(pa), _f64(ea)
        obs = np.empty((self.n, 18))
        rew = np.empty(self.n)
        done = np.empty(self.n, dtype=np.uint8)
        lib().orc_env_step_batch(self.envs, self.counts.ctypes.data_as(C.POINTER(C.c_int32)), self.n,
                                 _dp(self.M), _dp(pa), _dp(ea), _dp(obs), _dp(rew),
                                 done.ctypes.data_as(C.POINTER(C.c_uint8)), int(auto_reset), self.nthreads)
        return obs, rew, done

    def step_rk4(self, pa, ea, h=1.0, substeps=100, mu=MU_M, re=RE_M, j2=J2, auto_reset=True):
        pa, ea = _f64(pa), _f64(ea)
        obs = np.empty((self.n, 18))
        rew = np.empty(self.n)
        done = np.empty(self.n, dtype=np.uint8)
        lib().orc_env_step_rk4_batch(self.envs, self.counts.ctypes.data_as(C.POINTER(C.c_int32)), self.n,
                                     h, substeps, mu, re, j2, _dp(pa), _dp(ea), _dp(obs), _dp(rew),
                                     done.ctypes.data_as(C.POINTER(C.c_uint8)), int(auto_reset), self.nthreads)
        return obs, rew, done


# ------------------------------------------------------------------ normalisation (numpy, literal)
class RunningMeanStd:
    """normalization.py:7-29 (sequential Welford, n==1 rule Q7)."""

    def __init__(self, shape):
        self.n = 0
        self.mean = np.zeros(shape)
        self.S = np.zeros(shape)
        self.std = np.sqrt(self.S)

    def update(self, x):
        x = np.array(x, dtype=np.float64)
        self.n += 1
        if self.n == 1:
            self.mean = x
            self.std = x
        else:
            old_mean = self.mean.copy()
            self.mean = old_mean + (x - old_mean) / self.n
            self.S = self.S + (x - old_mean) * (x - self.mean)
            self.std = np.sqrt(self.S / self.n)


def chan_merge(n_a, mean_a, S_a, X):
    """Batched definition adopted for N>1 (SURVEY H7): merge the batch X [N, dim] into (n, mean, S)
    with Chan's parallel update; for N == 1 this is algebraically the Welford step of
    normalization.py:26-28."""
    X = np.asarray(X, dtype=np.float64)
    n_b = X.shape[0]
    mean_b = X.mean(axis=0)
    S_b = ((X - mean_b) ** 2).sum(axis=0)
    n = n_a + n_b
    delta = mean_b - mean_a
    mean = mean_a + delta * (n_b / n)
    S = S_a + S_b + delta * delta * (n_a * n_b / n)
    return n, mean, S


# ------------------------------------------------------------------ GAE
def gae(r, vs, vs_next, dw, done, gamma=0.99, lamda=0.95):
    r, vs, vs_next, dw, done = map(lambda a: _f32(a).ravel(), (r, vs, vs_next, dw, done))
    B = r.shape[0]
    adv = np.empty(B, dtype=np.float32)
    vt = np.empty(B, dtype=np.float32)
    lib().orc_gae(_fp(r), _fp(vs), _fp(vs_next), _fp(dw), _fp(done), B, gamma, lamda, _fp(adv), _fp(vt))
    return adv, vt


def gae_time_major(r, v, done, gamma=0.99, lamda=0.95):
    """r, done: [T, N]; v: [T+1, N] (v[t+1] is V(s') of step t; dw == done, Q8). Column-wise orc_gae."""
    T, N = r.shape
    adv = np.empty((T, N), dtype=np.float32)
    vt = np.empty((T, N), dtype=np.float32)
    for j in range(N):
        d = done[:, j].astype(np.float32)
        adv[:, j], vt[:, j] = gae(r[:, j], v[:-1, j], v[1:, j], d, d, gamma, lamda)
    return adv, vt


def adv_normalize(adv):
    a = _f32(adv).ravel().copy()
    lib().orc_adv_normalize(_fp(a), a.shape[0])
    return a.reshape(np.shape(adv))


# ------------------------------------------------------------------ actor / critic
def actor_forward(W, s, max_action=1.6):
    """W: dict with fc1.weight, fc1.bias, fc2.*, mean_layer.* (numpy fp32)."""
    s = _f32(s)
    n, in_dim = s.shape
    hid = W["fc1.weight"].shape[0]
    act = W["mean_layer.weight"].shape[0]
    mean = np.empty((n, act), dtype=np.float32)
    a = [_f32(W[k]) for k in ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "mean_layer.weight", "mean_layer.bias")]
    lib().orc_actor_forward(*[_fp(x) for x in a], in_dim, hid, act, max_action, _fp(s), n, _fp(mean))
    return mean


def critic_forward(W, s):
    s = _f32(s)
    n, in_dim = s.shape
    hid = W["fc1.weight"].shape[0]
    v = np.empty(n, dtype=np.float32)
    a = [_f32(W[k]) for k in ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias")]
    lib().orc_critic_forward(*[_fp(x) for x in a], in_dim, hid, _fp(s), n, _fp(v))
    return v


def gaussian_sample(mean, log_std, eps, max_action=1.6):
    mean, eps = _f32(mean), _f32(eps)
    log_std = _f32(log_std).ravel()
    n, act = mean.shape
    a = np.empty_like(mean)
    lp = np.empty_like(mean)
    lib().orc_gaussian_sample(_fp(mean), _fp(log_std), _fp(eps), n, act, max_action, _fp(a), _fp(lp))
    return a, lp
