"""Host logic of the opponent pool (no GPU): group bounds and their intersection with shards, the per-collect permutation,
the pool's FIFO ring and snapshot ids (library calls stubbed), and the shard-alignment precondition of VectorTrainer."""
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")


def _rollout():
    from ppo_rl_satellite_b200 import rollout
    return rollout


@pytest.mark.parametrize("n_total,groups", [(8192, 1), (8192, 4), (8192, 3), (65536 + 37, 8), (65536, 16), (1000, 16)])
def test_group_bounds(n_total, groups):
    R = _rollout()
    ends = R.pool_group_bounds(n_total, groups)
    tiles = -(-n_total // 128)
    assert len(ends) == groups and ends[-1] == n_total
    assert all(e % 128 == 0 for e in ends[:-1])
    assert all(b >= a for a, b in zip([0] + ends, ends))
    assert ends[:-1] == [min(128 * (tiles * k // groups), n_total) for k in range(1, groups)]
    sizes = np.diff([0] + ends)
    if tiles >= groups:                                   # equal up to one tile (and the ragged last one)
        assert sizes.min() > 0 and sizes.max() - sizes.min() <= 128


@pytest.mark.parametrize("world", [1, 2, 4, 8])
@pytest.mark.parametrize("groups", [1, 3, 8, 16])
def test_shard_groups_partition_every_shard(world, groups):
    R = _rollout()
    per = 4096
    ends = R.pool_group_bounds(world * per, groups)
    owner = np.repeat(np.arange(groups), np.diff([0] + ends))        # the group of every global row
    for rank in range(world):
        lo, hi = rank * per, (rank + 1) * per
        local = R.shard_groups(ends, lo, hi)
        loc_ends = [e for _, e in local]
        assert loc_ends[-1] == per and all(b > a for a, b in zip([0] + loc_ends, loc_ends))
        assert all(e % 128 == 0 for e in loc_ends[:-1])
        got = np.repeat([k for k, _ in local], np.diff([0] + loc_ends))
        assert np.array_equal(got, owner[lo:hi])


def test_permutation_depends_only_on_seed_and_collect_index():
    R = _rollout()
    for size in (1, 4, 16):
        p = R.pool_permutation(5, 3, size)
        assert sorted(p) == list(range(size))
        assert p == R.pool_permutation(5, 3, size) == R.pool_permutation(5 + 2 ** 64, 3, size)
    perms = {tuple(R.pool_permutation(5, c, 8)) for c in range(20)}
    assert len(perms) > 10                                        # varies with the collect index
    assert R.pool_permutation(6, 3, 8) != R.pool_permutation(5, 3, 8) or R.pool_permutation(6, 4, 8) != R.pool_permutation(5, 4, 8)


class _FakeLib:
    def __init__(self):
        self.snapshots = 0

    def sat_actor_tc_snapshot(self, w, image, tables, snap, stream):
        self.snapshots += 1
        return 0


@pytest.fixture()
def cpu_pool(monkeypatch):
    """OpponentPool on host tensors with the library stubbed: its ring and id bookkeeping only"""
    from ppo_rl_satellite_b200 import engine as eng
    fake = _FakeLib()
    monkeypatch.setattr(eng.L, "require_cuda", lambda: torch)
    monkeypatch.setattr(eng.L, "load", lambda: fake)
    monkeypatch.setattr(eng.L, "guard_device", lambda device: None)
    monkeypatch.setattr(eng.L, "stream_ptr", lambda: 0)
    return eng, fake


def _actor(value, use_tanh=1, max_action=1.6):
    from ppo_rl_satellite_b200 import _lib
    return types.SimpleNamespace(w=object(), critic=False, use_tanh=use_tanh, max_action=max_action,
                                 packed=torch.full((_lib.ACTOR_PACKED_FLOATS,), float(value)))


def test_pool_fifo_and_ids(cpu_pool):
    eng, fake = cpu_pool
    pool = eng.OpponentPool(3, device="cpu")
    assert len(pool) == 0 and pool.ids == []
    for v in range(5):
        assert pool.add(_actor(v)) == v
    assert len(pool) == 3 and pool.ids == [2, 3, 4] and fake.snapshots == 5
    assert [float(pool.kernel(k).packed[0]) for k in range(3)] == [2.0, 3.0, 4.0]    # slot k = the k-th oldest
    sd = pool.state_dict()
    other = eng.OpponentPool(4, device="cpu").load_state_dict(sd)
    assert other.ids == [2, 3, 4] and other.add(_actor(9)) == 5                       # ids go on after a reload
    assert [float(other.kernel(k).packed[0]) for k in range(4)] == [2.0, 3.0, 4.0, 9.0]
    with pytest.raises(eng.L.SatError):
        pool.add(_actor(0, use_tanh=0))
    with pytest.raises(eng.L.SatError):
        pool.add(_actor(0, max_action=1.0))
    with pytest.raises(eng.L.SatError):
        eng.OpponentPool(17, device="cpu")
    with pytest.raises(eng.L.SatError):
        eng.OpponentPool(2, device="cpu").load_state_dict(sd)                        # 3 snapshots do not fit


def test_misaligned_shards_are_refused():
    R = _rollout()
    env = types.SimpleNamespace(n=1000, device="cpu")
    with pytest.raises(R.eng.L.SatError, match="128-row"):
        R.VectorTrainer(env, None, None, 4, rank=1, world=2, opponent_pool=object())
