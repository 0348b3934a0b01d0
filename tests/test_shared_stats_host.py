"""CPU checks of statistics shared across ranks (sat_stats_fold): a numpy restatement of the two-pass fold over rank-major
per-block partials, checked against a direct mean / M2 of the union rows with ragged shards, and the host-side argument
checks and sizes of the new C entry points."""
import numpy as np
import pytest

from ppo_rl_satellite_b200 import _lib as L

THREADS = 256          # kMergeThreads: pass 1 and pass 2 are thread-strided over the global block index


def block_partials(x, rpb):
    """per-block (mean, M2) of x [n, dims], each block summed in row order (the env step's / norm_partial_kernel's tile)"""
    out = []
    for r0 in range(0, x.shape[0], rpb):
        t = x[r0:r0 + rpb]
        s = np.zeros(x.shape[1])
        for row in t:
            s = s + row
        mean = s / t.shape[0]
        m2 = np.zeros(x.shape[1])
        for row in t:
            d = row - mean
            m2 = m2 + d * d
        out.append(np.stack([mean, m2], axis=1))
    return np.array(out)                       # [blocks, dims, 2]


def block_sum_fixed(v):
    """warp xor tree then the 8 warp sums in warp order (block_sum_fixed in csrc/env_step.cu)"""
    v = np.array(v)
    for off in (16, 8, 4, 2, 1):
        v = v + v[np.arange(THREADS) ^ off]
    t = np.zeros(v.shape[1:])
    for w in range(THREADS // 32):
        t = t + v[32 * w]
    return t


def fold_ranks(gathered, rank_rows, rpb):
    """sat_stats_fold's merge over rank-major partials gathered [G, stride, dims, 2]: (N, grand mean, M2) per dim"""
    blocks = []                                # (rank, local block, rows) in global block order
    for r, m in enumerate(rank_rows):
        for j in range((m + rpb - 1) // rpb):
            blocks.append((r, j, min(rpb, m - j * rpb)))
    N = float(sum(rank_rows))
    dims = gathered.shape[2]
    wsum = np.zeros((THREADS, dims))
    for b, (r, j, nb) in enumerate(blocks):
        wsum[b % THREADS] = wsum[b % THREADS] + float(nb) * gathered[r, j, :, 0]
    grand = block_sum_fixed(wsum) / N
    m2 = np.zeros((THREADS, dims))
    for b, (r, j, nb) in enumerate(blocks):
        dm = gathered[r, j, :, 0] - grand
        m2[b % THREADS] = m2[b % THREADS] + (gathered[r, j, :, 1] + float(nb) * dm * dm)
    return N, grand, block_sum_fixed(m2)


def gather(shards, rpb):
    """rank-major [G, stride, dims, 2], each rank padded to the largest block count (padding is never read); a rank with
    no rows contributes no blocks"""
    stride = max((len(s) + rpb - 1) // rpb for s in shards)
    out = np.full((len(shards), stride, shards[0].shape[1], 2), np.nan)
    for r, s in enumerate(shards):
        if len(s):
            p = block_partials(s, rpb)
            out[r, :p.shape[0]] = p
    return out


@pytest.mark.parametrize("sizes,rpb", [((4096, 4096, 37), 64), ((8192, 4133), 64), ((4101, 4091), 64),
                                       ((1280, 1280, 1280, 1), 128), ((300, 0, 1000), 128), ((70000,), 64)])
def test_rank_major_fold_is_the_union_mean_and_m2(sizes, rpb):
    rng = np.random.default_rng(len(sizes) * 7 + sizes[0])
    dims = 5
    x = rng.normal(size=(sum(sizes), dims)) * np.array([1e5, 1.0, 3e3, 1e-3, 40.0]) + np.array([2e5, 0.0, -7e4, 1.0, 5.0])
    edges = np.cumsum((0,) + sizes)
    shards = [x[a:b] for a, b in zip(edges[:-1], edges[1:])]
    N, mean, m2 = fold_ranks(gather(shards, rpb), list(sizes), rpb)
    assert N == x.shape[0]
    ref_mean = x.mean(axis=0)
    ref_m2 = ((x - ref_mean) ** 2).sum(axis=0)
    assert np.allclose(mean, ref_mean, rtol=1e-13, atol=1e-12 * x.std(axis=0).max())
    assert np.allclose(m2, ref_m2, rtol=1e-11)


@pytest.mark.parametrize("sizes,rpb", [((4096, 4096, 37), 64), ((8192, 4133), 64), ((1280, 1280, 1280, 1), 128)])
def test_aligned_shards_fold_to_the_bits_of_the_union(sizes, rpb):
    """every shard but the last a multiple of the rows per block: the shards' blocks are the union's blocks, so the fold
    over G ranks and the fold over the union as one rank produce the same bits"""
    rng = np.random.default_rng(3)
    x = rng.normal(size=(sum(sizes), 4)) * 1e4 + 3e5
    edges = np.cumsum((0,) + sizes)
    shards = [x[a:b] for a, b in zip(edges[:-1], edges[1:])]
    got = fold_ranks(gather(shards, rpb), list(sizes), rpb)
    one = fold_ranks(gather([x], rpb), [x.shape[0]], rpb)
    assert got[0] == one[0] and np.array_equal(got[1], one[1]) and np.array_equal(got[2], one[2])


def test_partials_bytes_and_argument_checks():
    lib = L.load()
    assert lib.sat_stats_partials_bytes(4096, 0) == 64 * 19 * 2 * 8
    assert lib.sat_stats_partials_bytes(4097, 0) == 65 * 19 * 2 * 8
    assert lib.sat_stats_partials_bytes(4097, 18) == 33 * 18 * 2 * 8
    assert lib.sat_stats_partials_bytes(0, 0) == 0 and lib.sat_stats_partials_bytes(10, 33) == 0
    SAT_ERR_NULL, SAT_ERR_SIZE = -1, -2
    fake = 256                                 # never dereferenced: every case below is refused before a launch
    assert lib.sat_stats_fold(None, 1, 1, fake, 0, fake, None, None, fake, None) == SAT_ERR_NULL
    assert lib.sat_stats_fold(fake, 1, 1, None, 0, fake, None, None, fake, None) == SAT_ERR_NULL
    assert lib.sat_stats_fold(fake, 1, 1, fake, 0, fake, None, None, None, None) == SAT_ERR_NULL
    assert lib.sat_stats_fold(fake, 0, 1, fake, 0, fake, None, None, fake, None) == SAT_ERR_SIZE
    assert lib.sat_stats_fold(fake, 1, 0, fake, 0, fake, None, None, fake, None) == SAT_ERR_SIZE
    assert lib.sat_stats_fold(fake, 1, 1, fake, 33, fake, None, None, fake, None) == SAT_ERR_SIZE
    assert lib.sat_stats_fold(fake, 1, 1, fake, 18, fake, fake, None, fake, None) == SAT_ERR_SIZE
    assert lib.sat_stats_fold(fake, 1, 1, fake, 0, None, None, None, fake, None) == 0      # nothing to fold
    assert lib.sat_norm_partials(None, 10, 3, fake, fake, None) == SAT_ERR_NULL
    assert lib.sat_norm_partials(fake, 0, 3, fake, fake, None) == SAT_ERR_SIZE
    assert lib.sat_norm_partials(fake, 10, 33, fake, fake, None) == SAT_ERR_SIZE
    assert lib.sat_env_step_partials(None, fake, fake, None, None, None, None, fake, fake, None, fake, None, None) == SAT_ERR_NULL
