"""CPU checks of the GAE references: the oracle's orc_gae equals the reference's block (ppo_continuous.py:198-208, run
literally under numpy 2) bit for bit for any (gamma, lamda), and the vectorised time-major restatement that the GPU tests
use as their exact reference equals the oracle. No GPU needed."""
import numpy as np
import pytest

from gae_reference import F32, gae_scan, reference_block

PAIRS = [(0.99, 0.95), (0.99, 0.99), (0.98, 0.9), (0.995, 0.97), (1.0, 1.0), (0.9, 0.0)]
_rng = np.random.default_rng(20261022)
RANDOM_PAIRS = [(float(g), float(lam)) for g, lam in zip(_rng.uniform(0.9, 1.0, 20), _rng.uniform(0.8, 1.0, 20))]


def _bits(a):
    return np.ascontiguousarray(a, dtype=F32).view(np.uint32)


def _flat_inputs(seed, B, done_rate):
    rng = np.random.default_rng(seed)
    r = rng.normal(0, 2, B).astype(F32)
    vs = rng.normal(0, 5, B).astype(F32)
    vs_ = rng.normal(0, 5, B).astype(F32)
    done = (rng.random(B) < done_rate).astype(F32)
    dw = done * (rng.random(B) < 0.5).astype(F32)          # dw (terminal) implies done (episode end)
    return r, vs, vs_, dw, done


def test_literal_block_runs_in_float32():
    """NEP 50: a python float times an np.float32 stays float32, which is what makes the recursion an fp32 one"""
    assert int(np.__version__.split(".")[0]) >= 2
    assert type(0.99 * 0.95 * F32(1.5)) is np.float32
    adv, _ = reference_block(*_flat_inputs(0, 8, 0.0), 0.99, 0.95)
    assert adv.dtype == F32


@pytest.mark.parametrize("done_rate", [0.0, 0.02, 1.0])
@pytest.mark.parametrize("gamma,lamda", PAIRS + RANDOM_PAIRS)
def test_oracle_gae_equals_reference_block(oracle, gamma, lamda, done_rate):
    r, vs, vs_, dw, done = _flat_inputs(int(gamma * 1e6) ^ int(lamda * 1e6), 500, done_rate)
    ref_adv, ref_vt = reference_block(r, vs, vs_, dw, done, gamma, lamda)
    adv, vt = oracle.gae(r, vs, vs_, dw, done, gamma, lamda)
    assert np.array_equal(_bits(adv), _bits(ref_adv)), np.abs(adv - ref_adv).max()
    assert np.array_equal(_bits(vt), _bits(ref_vt))


def test_fp32_rounded_hyperparameters_are_not_the_reference():
    """the pairs above discriminate: gl = f32(f32(gamma) f32(lamda)) instead of f32(gamma lamda) changes the advantages"""
    r, vs, vs_, dw, done = _flat_inputs(5, 500, 0.02)
    ref_adv, _ = reference_block(r, vs, vs_, dw, done, 0.99, 0.99)
    gl_rounded = F32(float(F32(0.99)) * float(F32(0.99)))
    assert gl_rounded != F32(0.99 * 0.99)
    keep = F32(1) - done
    delta = (r + (F32(0.99) * (F32(1) - dw)) * vs_) - vs
    g, wrong = F32(0), np.empty_like(r)
    for t in range(499, -1, -1):
        g = delta[t] + (gl_rounded * g) * keep[t]
        wrong[t] = g
    assert not np.array_equal(wrong, ref_adv)


@pytest.mark.parametrize("T,N", [(1, 1), (1, 9), (7, 3), (64, 5), (65, 4), (130, 33)])
@pytest.mark.parametrize("gamma,lamda", [(0.99, 0.95), (0.99, 0.99), (0.995, 0.97), (0.9, 0.0)])
def test_time_major_restatement_equals_oracle(oracle, T, N, gamma, lamda):
    rng = np.random.default_rng(T * 1000 + N)
    r = rng.normal(0, 2, (T, N)).astype(F32)
    v = rng.normal(0, 5, (T + 1, N)).astype(F32)
    sc = rng.uniform(0.1, 2.0, T).astype(F32)
    for done in ((rng.random((T, N)) < 0.05).astype(np.uint8), np.ones((T, N), np.uint8), np.zeros((T, N), np.uint8)):
        adv, vt = gae_scan(r, v, done, gamma, lamda)
        o_adv, o_vt = oracle.gae_time_major(r, v, done, gamma, lamda)
        assert np.array_equal(_bits(adv), _bits(o_adv)) and np.array_equal(_bits(vt), _bits(o_vt))
        adv, vt = gae_scan(r, v, done.astype(bool), gamma, lamda, r_scale=sc)
        o_adv, o_vt = oracle.gae_time_major(r * sc[:, None], v, done, gamma, lamda)
        assert np.array_equal(_bits(adv), _bits(o_adv)) and np.array_equal(_bits(vt), _bits(o_vt))
