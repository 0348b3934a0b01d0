"""The advantage stage after every rollout (VectorTrainer.compute_advantages): critic values (sat_critic_forward), the
time-major GAE scan (sat_gae), the advantage moments (sat_adv_moments) and the in-place normalisation
(sat_adv_normalize), each against an exact or fp64 reference at the shapes and edges where the kernels branch:

- GAE bit for bit against the fp32 restatement (tests/gae_reference.py) for every envs-per-CTA instantiation and its
  boundaries (8 envs below N = 4736, 16 up to 28 415, 32 from 28 416), partial top tiles, done on the tile edges,
  r_scale and non-default (gamma, lamda); inputs are prefixes of NaN-filled buffers and outputs views between sentinels;
- the moments against exact sums, on the float4 path, its scalar tail and the misaligned scalar path;
- the normalisation against fp64 within the bound that follows from the kernel's fp32 mean and denominator;
- the critic against a torch fp64 forward, tanh and ReLU, ragged row counts, written into a view of the values buffer;
- the whole stage inside a VectorTrainer rollout."""
import math

import numpy as np
import pytest

from gae_reference import F32, gae_fp64, gae_scan

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24                 # unit roundoff of fp32
PAD = 4099                       # elements of NaN / sentinel around every buffer
SENTINEL = -31337.25


@pytest.fixture(scope="module")
def eng():
    from ppo_rl_satellite_b200 import engine
    return engine


@pytest.fixture(scope="module")
def lib_errors():
    from ppo_rl_satellite_b200 import _lib
    return _lib.SatError


def _bits(a):
    return np.ascontiguousarray(a, dtype=F32).view(np.uint32)


def _in_nan_prefix(a):
    """a device copy of `a` that is the prefix of a buffer whose tail is NaN (0xff for bytes): a read past the end of the
    operand poisons the result"""
    a = torch.as_tensor(np.ascontiguousarray(a))
    fill = float("nan") if a.dtype.is_floating_point else 255
    buf = torch.full((a.numel() + PAD,), fill, dtype=a.dtype, device="cuda")
    view = buf[:a.numel()].view(a.shape)
    view.copy_(a)
    return view


class _Sentinelled:
    """an fp32 output `shape` at offset `off` of a buffer whose other elements hold SENTINEL"""

    def __init__(self, shape, off=PAD):
        n = int(np.prod(shape))
        self.buf = torch.full((n + off + PAD,), SENTINEL, dtype=torch.float32, device="cuda")
        self.off, self.n = off, n
        self.view = self.buf[off:off + n].view(shape)

    def assert_sentinels(self):
        b = self.buf.cpu().numpy()
        assert (b[:self.off] == SENTINEL).all() and (b[self.off + self.n:] == SENTINEL).all(), "write outside the output"


def _done_pattern(kind, T, N, rng):
    if kind == "none":
        return np.zeros((T, N), np.uint8)
    if kind == "all":
        return np.ones((T, N), np.uint8)
    if kind == "random":
        return (rng.random((T, N)) < 0.03).astype(np.uint8)
    t = np.arange(T)[:, None]                                   # "edges": done on the first and last row of each tile
    return np.broadcast_to(((t % 64 == 0) | (t % 64 == 63)).astype(np.uint8), (T, N)).copy()


def _r_scale(rng, T):
    """as the rollout builds it: (1 / (ret_std + 1e-8)).float() from the fp64 running return std"""
    ret_std = torch.from_numpy(rng.uniform(0.05, 3.0, T))
    return (1.0 / (ret_std + 1e-8)).float().numpy()


def _run_gae(eng, r, v, done, gamma, lamda, r_scale):
    T, N = r.shape
    a, vt = _Sentinelled((T, N)), _Sentinelled((T, N))
    sc = _in_nan_prefix(r_scale) if r_scale is not None else None
    out = eng.gae_time_major(_in_nan_prefix(r), _in_nan_prefix(v), _in_nan_prefix(done), gamma, lamda, r_scale=sc,
                             adv=a.view, v_target=vt.view)
    assert out[0] is a.view and out[1] is vt.view
    a.assert_sentinels(); vt.assert_sentinels()
    return a.view.cpu().numpy(), vt.view.cpu().numpy()


# ============================================================================ GAE, exact
GAE_N = [1, 4735, 4736, 8192, 28415, 28416, 65573]
GAE_T = [1, 63, 64, 65, 129]
GL_PAIRS = [(0.99, 0.95), (0.99, 0.99), (0.995, 0.97), (0.98, 0.9)]


@pytest.mark.parametrize("T", GAE_T)
@pytest.mark.parametrize("N", GAE_N)
def test_gae_bit_identical_to_restatement(eng, N, T):
    """every tiling and its boundaries, partial and whole top tiles, four done patterns, with and without r_scale, the
    default and three other (gamma, lamda)"""
    rng = np.random.default_rng(N * 1000 + T)
    r = rng.normal(0, 2, (T, N)).astype(F32)
    v = rng.normal(0, 5, (T + 1, N)).astype(F32)
    for k, kind in enumerate(("none", "all", "random", "edges")):
        done = _done_pattern(kind, T, N, rng)
        for j, sc in enumerate((None, _r_scale(rng, T))):
            gamma, lamda = GL_PAIRS[(2 * k + j) % len(GL_PAIRS)]
            adv, vt = _run_gae(eng, r, v, done, gamma, lamda, sc)
            ref_adv, ref_vt = gae_scan(r, v, done, gamma, lamda, r_scale=sc)
            bad = np.flatnonzero(_bits(adv) != _bits(ref_adv))
            assert bad.size == 0, (kind, sc is not None, gamma, lamda, bad[:5], np.abs(adv - ref_adv).max())
            assert np.array_equal(_bits(vt), _bits(ref_vt)), (kind, sc is not None, gamma, lamda)


@pytest.mark.parametrize("gamma,lamda", [(0.99, 0.95), (0.99, 0.99)])
def test_gae_config5_shard_bit_identical(eng, gamma, lamda):
    """the config-5 shard (T = 2048, N = 8192: the 16-env form, 32 whole tiles) with r_scale and 3 % dones"""
    T, N = 2048, 8192
    rng = np.random.default_rng(5)
    r = rng.normal(0, 2, (T, N)).astype(F32)
    v = rng.normal(0, 5, (T + 1, N)).astype(F32)
    done = (rng.random((T, N)) < 0.03).astype(np.uint8)
    sc = _r_scale(rng, T)
    adv, vt = _run_gae(eng, r, v, done, gamma, lamda, sc)
    ref_adv, ref_vt = gae_scan(r, v, done, gamma, lamda, r_scale=sc)
    assert np.array_equal(_bits(adv), _bits(ref_adv)) and np.array_equal(_bits(vt), _bits(ref_vt))


def test_gae_bool_done_equals_uint8(eng):
    rng = np.random.default_rng(3)
    T, N = 65, 4736
    r = torch.from_numpy(rng.normal(0, 2, (T, N)).astype(F32)).cuda()
    v = torch.from_numpy(rng.normal(0, 5, (T + 1, N)).astype(F32)).cuda()
    d = torch.from_numpy(rng.random((T, N)) < 0.1).cuda()
    a8, t8 = eng.gae_time_major(r, v, d.to(torch.uint8), 0.99, 0.99)
    ab, tb = eng.gae_time_major(r, v, d, 0.99, 0.99)
    assert torch.equal(a8.view(torch.int32), ab.view(torch.int32)) and torch.equal(t8.view(torch.int32), tb.view(torch.int32))


# ============================================================================ GAE against fp64
@pytest.mark.parametrize("N,T,gamma,lamda,kind", [(4735, 129, 0.99, 0.95, "random"), (28416, 65, 0.995, 0.97, "none"),
                                                  (65573, 64, 0.98, 0.9, "edges"), (8192, 2048, 0.99, 0.99, "random"),
                                                  (1, 129, 1.0, 1.0, "none")])
def test_gae_restatement_within_fp64_bound(eng, N, T, gamma, lamda, kind):
    """the exact reference (and so the kernel) against fp64 GAE with gl = gamma lamda. Each step of the fp32 recursion
    rounds the delta (3 operations on |r| + |v'| + |v|, plus gamma rounded to fp32), the product and the sum (on |delta| +
    |g|) and uses gl rounded to fp32; those local errors decay by gamma lamda per step, so the total is at most
    4 u max(|r| + |v'| + |v| + |g|) min(T, 1 / (1 - gamma lamda)). Swapped gamma / lamda or a dropped r_scale on both sides
    of the exact comparison would be caught here."""
    rng = np.random.default_rng(N + T)
    r = rng.normal(0, 2, (T, N)).astype(F32)
    v = rng.normal(0, 5, (T + 1, N)).astype(F32)
    done = _done_pattern(kind, T, N, rng)
    sc = _r_scale(rng, T)
    adv, _ = _run_gae(eng, r, v, done, gamma, lamda, sc)
    ref, _ = gae_scan(r, v, done, gamma, lamda, r_scale=sc)
    assert np.array_equal(_bits(adv), _bits(ref))
    adv64, _ = gae_fp64(r, v, done, gamma, lamda, r_scale=sc)
    rs = np.abs(r.astype(np.float64) * sc[:, None])
    mag = (rs + np.abs(v[1:]) + np.abs(v[:-1]) + np.abs(adv64)).max()
    horizon = T if gamma * lamda >= 1.0 else min(T, 1.0 / (1.0 - gamma * lamda))
    bound = 4 * U32 * mag * horizon
    err = np.abs(adv.astype(np.float64) - adv64).max()
    assert err <= bound, (err, bound)
    assert err > 0 or kind == "all"                             # the fp32 recursion does round


# ============================================================================ moments
BIG = 1184 * 256 * 4 * 4          # elements one float4 pass of the partial kernel covers (4 loads per thread)
COUNTS = [1, 2, 3, 4, 5, 255, 256, 257, BIG - 1, BIG + 1, 2 ** 24 + 3]


def _exact_sums(x):
    """sum and sum of squares of fp32 values: the squares are exact in fp64; extended-precision pairwise sums are far
    below the tested bound (math.fsum where long double is plain double)"""
    x64 = x.astype(np.float64)
    if np.finfo(np.longdouble).eps < 1e-18:
        xl = x64.astype(np.longdouble)
        return float(xl.sum()), float((xl * xl).sum()), float(np.abs(xl).sum())
    return math.fsum(x64), math.fsum(x64 * x64), math.fsum(np.abs(x64))


def _values(count, shifted, seed):
    x = np.random.default_rng(seed).standard_normal(count)
    return (x + 1e4 if shifted else x).astype(F32)


def _at_offset(x, off):
    """x written at float offset `off` (0..3) of a sentinel-filled device buffer: off != 0 makes the pointer 4-, 8- or
    12-byte aligned (the partial kernel's scalar path); off = 0 keeps it 16-byte aligned (float4 path + scalar tail)"""
    s = _Sentinelled((x.size,), off=off)
    s.view.copy_(torch.from_numpy(x))
    return s


@pytest.mark.parametrize("shifted", [False, True], ids=["n01", "1e4+n01"])
@pytest.mark.parametrize("count", COUNTS)
def test_adv_moments_exact_sums(eng, count, shifted):
    x = _values(count, shifted, count)
    s1, s2, sabs = _exact_sums(x)
    for off in range(4):
        s = _at_offset(x, off)
        m = eng.adv_moments(s.view).cpu().numpy()
        assert m[2] == count
        assert abs(m[0] - s1) <= 1e-13 * sabs, (off, m[0], s1)
        assert abs(m[1] - s2) <= 1e-13 * s2, (off, m[1], s2)
        s.assert_sentinels()


# ============================================================================ normalisation
def _normalize_bound(x, count_total, s1, s2):
    """fp64 (x - mu) / (sigma + 1e-5) of the fp32 inputs and a per-element bound on the kernel's result. The kernel forms
    m = f32(mean) and den = f32(f32(sqrt(var)) + 1e-5) from fp64 moments (each within 1e-13 of exact, as tested above, so
    the one-pass variance is within 4e-13 S2 / (n - 1)), then rounds x - m and the quotient:
        |y - y*| <= e_m / den + |x - mu| e_den / (den (den - e_den)) + 2 u |x - mu| / den + 2 u e_m / den"""
    n = float(count_total)
    mu = s1 / n
    var = max((s2 - n * mu * mu) / (n - 1.0), 0.0)
    sd = math.sqrt(var)
    den = sd + 1e-5
    x64 = x.astype(np.float64)
    e_m = U32 * abs(mu) + 1e-13 * abs(s1) / n + 1e-300
    e_var = 4e-13 * s2 / (n - 1.0)
    e_sd = min(e_var / sd if sd > 0 else math.inf, math.sqrt(e_var))
    e_den = U32 * sd + e_sd + U32 * den
    assert e_den < 0.5 * den
    d = np.abs(x64 - mu)
    bound = e_m / den + d * e_den / (den * (den - e_den)) + 2 * U32 * (d + e_m) / den
    return (x64 - mu) / den, 2.0 * bound


@pytest.mark.parametrize("shifted", [False, True], ids=["n01", "1e4+n01"])
@pytest.mark.parametrize("count", COUNTS[1:])
def test_adv_normalize_within_bound(eng, count, shifted):
    x = _values(count, shifted, count + 1)
    s1, s2, _ = _exact_sums(x)
    want, bound = _normalize_bound(x, count, s1, s2)
    for off in range(4):
        s = _at_offset(x, off)
        eng.adv_normalize_(s.view, group=False)
        y = s.view.cpu().numpy().astype(np.float64)
        s.assert_sentinels()
        excess = np.abs(y - want) - bound
        assert excess.max() <= 0, (off, int(excess.argmax()), float(np.abs(y - want).max()))


@pytest.mark.parametrize("value", [3.5, 0.1, 1e4 + 0.3, -7.0])
@pytest.mark.parametrize("count", [2, 5, 257, BIG + 1])
def test_adv_normalize_constant_input_is_zero(eng, value, count):
    """zero variance: x - f32(mean) is exactly 0 (the fp64 mean of n equal fp32 values rounds back to the value), and the
    denominator is 1e-5, not 0"""
    s = _at_offset(np.full(count, value, dtype=F32), count % 4)
    eng.adv_normalize_(s.view, group=False)
    y = s.view.cpu().numpy()
    s.assert_sentinels()
    assert not np.isnan(y).any() and np.array_equal(_bits(y), np.zeros(count, np.uint32))


def test_adv_normalize_single_element_is_nan_like_torch_std(eng):
    for off in range(4):
        s = _at_offset(np.array([2.5], dtype=F32), off)
        eng.adv_normalize_(s.view, group=False)
        s.assert_sentinels()
        assert torch.isnan(s.view).all()
    with pytest.warns(UserWarning, match="degrees of freedom"):
        assert torch.isnan(torch.tensor([2.5]).std())


@pytest.mark.parametrize("count", [257, BIG + 1])
def test_adv_normalize_halves_with_caller_sums_equal_union(eng, count):
    """two shards add their moments (what the all-reduce does) and each normalises its half like the union buffer"""
    x = _values(count, True, 77)
    h = count // 2 + 1                                          # an odd split: the second half starts misaligned
    a = _at_offset(x[:h], 0)
    b2 = _Sentinelled((count - h,), off=h % 4)
    b2.view.copy_(torch.from_numpy(x[h:]))
    sums = eng.adv_moments(a.view) + eng.adv_moments(b2.view)
    assert sums[2].item() == count
    eng.adv_normalize_(a.view, sums=sums.clone(), group=False)
    eng.adv_normalize_(b2.view, sums=sums.clone(), group=False)
    whole = _at_offset(x, 0)
    eng.adv_normalize_(whole.view, group=False)
    s1, s2, _ = _exact_sums(x)
    want, bound = _normalize_bound(x, count, s1, s2)
    y = np.concatenate([a.view.cpu().numpy(), b2.view.cpu().numpy()]).astype(np.float64)
    assert (np.abs(y - want) <= bound).all()
    assert (np.abs(whole.view.cpu().numpy() - want) <= bound).all()
    for s in (a, b2, whole):
        s.assert_sentinels()


# ============================================================================ critic values
def _critic_weights(seed, boost):
    """orthogonal init as the reference's Critic (ppo_continuous.py:66-80), plus small random biases so the bias terms
    count; boost scales every layer"""
    g = torch.Generator().manual_seed(seed)
    w = {}
    for name, (o, i) in (("fc1", (256, 18)), ("fc2", (256, 256)), ("fc3", (1, 256))):
        m = torch.empty(o, i)
        torch.nn.init.orthogonal_(m, generator=g)
        w[f"{name}.weight"] = m * boost
        w[f"{name}.bias"] = 0.1 * boost * torch.randn(o, generator=g)
    return w


def _critic_torch(w, obs, dtype, use_tanh):
    act = torch.tanh if use_tanh else torch.relu
    p = {k: t.to(device=obs.device, dtype=dtype) for k, t in w.items()}
    x = obs.to(dtype)
    h = act(x @ p["fc1.weight"].T + p["fc1.bias"])
    h = act(h @ p["fc2.weight"].T + p["fc2.bias"])
    return (h @ p["fc3.weight"].T + p["fc3.bias"]).reshape(-1)


def _check_values(v, obs, w, use_tanh, groups):
    """|v - v64| <= 4 max|v_torch32 - v64| + 1e-6 max|v64|, per group of rows of similar scale"""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        v64 = _critic_torch(w, obs, torch.float64, use_tanh)
        v32 = _critic_torch(w, obs, torch.float32, use_tanh).double()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    for rows in groups:
        if rows.numel() == 0:
            continue
        ref = v64[rows]
        err = (v[rows].double() - ref).abs().max().item()
        bound = 4 * (v32[rows] - ref).abs().max().item() + 1e-6 * ref.abs().max().item()
        assert err <= bound, (err, bound)


@pytest.mark.parametrize("boost", [1.0, 3.0], ids=["orthogonal", "boosted"])
@pytest.mark.parametrize("use_tanh", [1, 0], ids=["tanh", "relu"])
def test_critic_values_against_fp64(eng, use_tanh, boost):
    w = _critic_weights(11 + use_tanh, boost)
    critic = eng.GaussianActorKernel(use_tanh=bool(use_tanh), critic=True).load_state_dict(w)
    gen = torch.Generator(device="cuda").manual_seed(int(boost * 10) + use_tanh)
    for n in (1, 63, 64, 65, 4097, 66 * 8192 + 37):
        obs = torch.randn(n, 18, device="cuda", generator=gen)
        big = torch.arange(0, n, 97, device="cuda")            # every 97th row at |x| ~ 50
        obs[big] = 50.0 * torch.sign(obs[big]) + torch.randn(big.numel(), 18, device="cuda", generator=gen)
        is_big = torch.zeros(n, dtype=torch.bool, device="cuda")
        is_big[big] = True
        groups = (torch.nonzero(~is_big).reshape(-1), big)
        _check_values(critic.value(obs), obs, w, use_tanh, groups)
        # into row 1 of a [T + 1, n] values buffer, as compute_advantages writes it: rows 0 and 2 stay untouched
        vals = torch.full((3, n), SENTINEL, device="cuda")
        assert critic.value(obs, out=vals[1]) is not None
        assert (vals[0] == SENTINEL).all() and (vals[2] == SENTINEL).all()
        _check_values(vals[1], obs, w, use_tanh, groups)
        if n == 4097:                                          # obs / out as views of the flattened [T + 1, n] buffers
            obs3 = obs.repeat(3, 1).view(3, n, 18)
            flat = _Sentinelled((3 * n,))
            critic.value(obs3.view(-1, 18), out=flat.view)
            flat.assert_sentinels()
            assert torch.equal(flat.view.view(3, n)[2], vals[1])


# ============================================================================ end to end
def _args(n, T):
    import types
    return types.SimpleNamespace(policy_dist="Gaussian", max_action=1.6, batch_size=n * T, mini_batch_size=512,
                                 max_train_steps=int(3e6), lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1,
                                 K_epochs=2, entropy_coef=0.01, set_adam_eps=True, use_grad_clip=True, use_lr_decay=True,
                                 use_adv_norm=True, state_dim=18, action_dim=3, hidden_width=256, use_tanh=1,
                                 use_orthogonal_init=True, chkpt_dir="/tmp")


@pytest.mark.parametrize("n,lamda", [(4736, 0.95), (28416, 0.97)])
def test_vector_trainer_advantage_stage(eng, monkeypatch, n, lamda):
    """a real rollout (running statistics on, so r_scale is used) through compute_advantages: critic values, GAE before
    the normalisation, v_target, the normalised advantages and the explained variance, each against its reference"""
    from ppo_rl_satellite_b200 import rollout
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    T = 65
    torch.manual_seed(0)
    env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=5, auto_reset=True)
    agent, opp = P.PPO_continuous(_args(n, T), "pursuer"), P.PPO_continuous(_args(n, T), "evader")
    agent.lamda = lamda
    assert agent.use_adv_norm
    tr = rollout.VectorTrainer(env, agent, opp, T)
    assert tr.ret_stats is not None
    tr.collect()
    buf = tr.buf
    rew64, done, ret_std, obs = (t.clone() for t in (buf.rew64, buf.done, buf.ret_std, buf.obs))
    assert done.any()
    seen = {}
    real = eng.adv_normalize_

    def spy(adv, *a, **k):
        seen["adv"] = adv.clone()
        return real(adv, *a, **k)
    monkeypatch.setattr(eng, "adv_normalize_", spy)
    tr.compute_advantages(explained_variance=True)

    w = {k: t.detach().cpu() for k, t in agent.critic.state_dict().items()}
    _check_values(buf.values.view(-1), obs.view(-1, 18), w, 1, (torch.arange((T + 1) * n, device="cuda"),))
    values = buf.values.cpu().numpy()
    r32 = rew64.float().cpu().numpy()
    sc = (1.0 / (ret_std + 1e-8)).float().cpu().numpy()
    ref_adv, ref_vt = gae_scan(r32, values, done.cpu().numpy(), agent.gamma, agent.lamda, r_scale=sc)
    adv0 = seen["adv"].cpu().numpy()
    assert np.array_equal(_bits(adv0), _bits(ref_adv))
    assert np.array_equal(_bits(buf.v_target.cpu().numpy()), _bits(ref_vt))

    x = adv0.ravel()
    s1, s2, _ = _exact_sums(x)
    want, bound = _normalize_bound(x, x.size, s1, s2)
    assert (np.abs(buf.adv.cpu().numpy().ravel().astype(np.float64) - want) <= bound).all()

    a64, t64 = adv0.astype(np.float64), ref_vt.astype(np.float64)
    ev = 1.0 - np.var(a64) / np.var(t64)
    got = tr.explained_variance.item()
    assert abs(got - ev) <= 1e-9 * max(1.0, abs(ev)), (got, ev)


# ============================================================================ argument checks
def test_gae_time_major_rejects_bad_arguments(eng, lib_errors):
    T, N = 5, 7
    r = torch.zeros(T, N, device="cuda")
    v = torch.zeros(T + 1, N, device="cuda")
    d = torch.zeros(T, N, dtype=torch.uint8, device="cuda")
    sc = torch.ones(T, device="cuda")
    eng.gae_time_major(r, v, d, r_scale=sc)                     # the well-formed call runs
    bad = [
        dict(r=torch.zeros(T * N, device="cuda")),                       # r not [T, N]
        dict(v=torch.zeros(T, N, device="cuda")),                        # v [T, N]: the kernel would read v[T N + e]
        dict(v=torch.zeros(T + 2, N, device="cuda")),
        dict(v=torch.zeros(T + 1, N + 1, device="cuda")),
        dict(done=torch.zeros(T, N + 1, dtype=torch.uint8, device="cuda")),
        dict(done=torch.zeros(T, N, dtype=torch.float32, device="cuda")),
        dict(done=torch.zeros(T, N, dtype=torch.int32, device="cuda")),
        dict(r_scale=torch.ones(T + 1, device="cuda")),
        dict(r_scale=torch.ones(T, dtype=torch.float64, device="cuda")),
        dict(r=torch.zeros(T, N, dtype=torch.float64, device="cuda")),
        dict(v=torch.zeros(T + 1, N, dtype=torch.float16, device="cuda")),
        dict(adv=torch.zeros(T, N + 1, device="cuda")),
        dict(v_target=torch.zeros(T, N, dtype=torch.float64, device="cuda")),
        dict(v=torch.zeros(T + 1, N)),                                   # host tensor
        dict(done=torch.zeros(T, N, dtype=torch.uint8)),
        dict(r_scale=torch.ones(T)),
    ]
    for kw in bad:
        args = dict(r=r, v=v, done=d, r_scale=sc)
        args.update(kw)
        rr, vv, dd = args.pop("r"), args.pop("v"), args.pop("done")
        with pytest.raises(lib_errors):
            eng.gae_time_major(rr, vv, dd, **args)


def test_critic_value_rejects_bad_arguments(eng, lib_errors):
    critic = eng.GaussianActorKernel(critic=True).load_state_dict(_critic_weights(1, 1.0))
    obs = torch.zeros(9, 18, device="cuda")
    critic.value(obs)
    for o in (torch.zeros(9, 17, device="cuda"), torch.zeros(9 * 18, device="cuda"),
              torch.zeros(9, 18, dtype=torch.float64, device="cuda"), torch.zeros(9, 18)):
        with pytest.raises(lib_errors):
            critic.value(o)
    for out in (torch.zeros(8, device="cuda"), torch.zeros(9, 1, device="cuda"),
                torch.zeros(9, dtype=torch.float64, device="cuda"), torch.zeros(9)):
        with pytest.raises(lib_errors):
            critic.value(obs, out=out)
    with pytest.raises(lib_errors):
        eng.GaussianActorKernel().load_state_dict(_actor_weights()).value(obs)


def _actor_weights():
    g = torch.Generator().manual_seed(2)
    return {"fc1.weight": torch.randn(256, 18, generator=g), "fc1.bias": torch.zeros(256),
            "fc2.weight": torch.randn(256, 256, generator=g), "fc2.bias": torch.zeros(256),
            "mean_layer.weight": torch.randn(3, 256, generator=g), "mean_layer.bias": torch.zeros(3),
            "log_std": torch.zeros(1, 3)}
