"""Batched on-device rollout + PPO update (BASELINE config 5): N envs x T steps per GPU, everything resident in HBM.

Per step: pursuer actor kernel (observation rebuilt + normalised from the fp64 state, Philox sample) -> evader actor
kernel -> fused env step (statistics updated in-kernel). After T steps: critic values, time-major GAE kernel,
advantage normalisation with all-reduced moments, then the K-epoch minibatch update (fused forward/backward/Adam kernels,
or the PyTorch step, + NCCL gradient all-reduce). Envs shard across ranks with no traffic during the rollout (SURVEY.md s8e)."""
from __future__ import annotations

import numpy as np
import torch

from . import engine as eng

POOL_TILE = 128            # rows per tile of the pool launch: every group bound but the last is a multiple of it


def pool_group_bounds(n_total: int, groups: int):
    """exclusive ends of `groups` contiguous groups over n_total global rows: 128 floor(tiles k / groups) for k = 1 ..
    groups with tiles = ceil(n_total / 128), the last = n_total (a group may be empty when there are fewer tiles than
    groups)"""
    tiles = -(-int(n_total) // POOL_TILE)
    ends = [min(POOL_TILE * (tiles * k // groups), int(n_total)) for k in range(1, groups + 1)]
    ends[-1] = int(n_total)
    return ends


def shard_groups(ends, lo: int, hi: int):
    """the groups (global bounds `ends`) that hold rows of the shard [lo, hi): [(group index, group end in shard rows)]"""
    out, start = [], 0
    for k, e in enumerate(ends):
        a, b = max(start, lo), min(e, hi)
        if b > a:
            out.append((k, b - lo))
        start = e
    return out


def pool_permutation(seed: int, collect_index: int, size: int):
    """which pool slot plays group k: a permutation drawn from (seed, collect index) only, the same on every rank"""
    rng = np.random.default_rng([int(seed) & (2 ** 64 - 1), int(collect_index)])
    return [int(v) for v in rng.permutation(size)]


class RolloutBuffer:
    """time-major device storage; s_ is implicit (obs[t+1]) because done == dw in this env (SURVEY Q8)."""

    def __init__(self, T: int, n: int, device="cuda"):
        self.T, self.n = T, n
        d = torch.device(device)
        self.obs = torch.empty((T + 1, n, 18), dtype=torch.float32, device=d)
        self.act = torch.empty((T, n, 3), dtype=torch.float32, device=d)
        self.logp = torch.empty((T, n, 3), dtype=torch.float32, device=d)
        self.opp_act = torch.empty((T, n, 3), dtype=torch.float32, device=d)
        self.opp_logp = torch.empty((T, n, 3), dtype=torch.float32, device=d)
        self.rew64 = torch.empty((T, n), dtype=torch.float64, device=d)
        self.done = torch.empty((T, n), dtype=torch.uint8, device=d)
        self.ret_std = torch.ones(T, dtype=torch.float64, device=d)
        self.values = torch.empty((T + 1, n), dtype=torch.float32, device=d)
        self.adv = torch.empty((T, n), dtype=torch.float32, device=d)
        self.v_target = torch.empty((T, n), dtype=torch.float32, device=d)

    @property
    def bytes_per_sample(self):
        return 18 * 4 + 4 * 3 * 4 + 8 + 1 + 3 * 4


class VectorTrainer:
    """Drives `agent` (learner: pursuer for flag 0, evader for flag 1) against `opponent` on an EnvBatch.

    stats_group (a torch.distributed process group, default None): the ranks of the group each drive their shard of one
    env batch, and the running statistics (observation normaliser, return statistics behind the reward scaling) are
    shared: the initial observations' statistics and every collect() step fold every rank's shard (EnvBatch.share_stats,
    RunningStats.update_normalize with group). Every rank then holds the same statistics, those of the union batch, bit
    for bit when every rank but the last holds a multiple of 128 envs (the initial observations are folded in blocks of
    128 rows, the steps in blocks of 64) and the env batches key their starts by global env index (row_offset). Collective: every rank of the group builds its trainer
    with the same stats_group. None: each rank's statistics see its own shard only.

    opponent_pool (engine.OpponentPool, default None): the learner plays past snapshots of the opponent instead of its
    current weights. Every collect() splits the global rows (world shards of env.n) into len(pool) groups with
    pool_group_bounds, gives group k the snapshot in slot pool_permutation(seed, collect index)[k] and samples this
    shard's groups in the learner's launch (sample_vs_pool); it then sets opponent_stats, per group of the shard: the
    snapshot id, the rows, the learner's mean reward and the episodes finished. With world > 1 every shard must start on a
    128-row boundary. None: the opponent's current weights on every row (sample_pair)."""

    def __init__(self, env: eng.EnvBatch, agent, opponent, T: int, use_state_norm=True, use_reward_scaling=True,
                 rank: int = 0, seed: int = 0, strict_errors: bool = False, stats_group=None, opponent_pool=None,
                 world: int = 1):
        if opponent_pool is not None and int(world) > 1 and (rank * env.n) % POOL_TILE:
            raise eng.L.SatError(f"an opponent pool over {world} shards needs every shard to start on a {POOL_TILE}-row "
                                 f"boundary (row offset {rank * env.n})")
        self.env, self.agent, self.opponent, self.T = env, agent, opponent, T
        self.strict_errors = strict_errors
        self.buf = RolloutBuffer(T, env.n, env.device)
        self.obs_stats = eng.RunningStats(18, env.device) if use_state_norm else None
        self.ret_stats = eng.RunningStats(1, env.device) if use_reward_scaling else None
        self.row_offset = rank * env.n            # the global row id of env 0 only when every shard holds env.n envs
        self.seed = seed
        self.t_global = 0
        self.world, self.opponent_pool, self.collects, self.opponent_stats = int(world), opponent_pool, 0, None
        self.explained_variance = None
        if stats_group is not None:
            env.share_stats(stats_group)
        if self.obs_stats is not None:
            self.obs_stats.update_normalize(env.observe(), group=stats_group)   # statistics of the initial observations
        self.learner_is_pursuer = env.params.flag == 0

    def collect(self):
        env, buf = self.env, self.buf
        if self.agent._dirty:
            self.agent.sync_kernels()
        if self.opponent._dirty:
            self.opponent.sync_kernels()
        pool = self.opponent_pool
        if pool is not None:
            if len(pool) == 0:
                raise eng.L.SatError("the opponent pool is empty")
            local = shard_groups(pool_group_bounds(self.world * env.n, len(pool)), self.row_offset, self.row_offset + env.n)
            perm = pool_permutation(self.seed, self.collects, len(pool))
            slots, ends = [perm[k] for k, _ in local], [e for _, e in local]
        for t in range(self.T):
            g = self.t_global
            # learner and opponent act on the same observation (CPPO_main.py:122-123): one launch for both networks
            if pool is None:
                self.agent.actor_kernel.sample_pair(self.opponent.actor_kernel, env=env, obs_stats=self.obs_stats,
                                                    seed=self.seed, step=2 * g, other_step=2 * g + 1, row_offset=self.row_offset,
                                                    act=buf.act[t], logp=buf.logp[t], obs_out=buf.obs[t],
                                                    other_act=buf.opp_act[t], other_logp=buf.opp_logp[t])
            else:
                self.agent.actor_kernel.sample_vs_pool(pool, slots, ends, env=env, obs_stats=self.obs_stats, seed=self.seed,
                                                       step=2 * g, other_step=2 * g + 1, row_offset=self.row_offset,
                                                       act=buf.act[t], logp=buf.logp[t], obs_out=buf.obs[t],
                                                       other_act=buf.opp_act[t], other_logp=buf.opp_logp[t])
            pa, ea = (buf.act[t], buf.opp_act[t]) if self.learner_is_pursuer else (buf.opp_act[t], buf.act[t])
            env.step(pa, ea, reward=buf.rew64[t], done=buf.done[t], obs_stats=self.obs_stats, ret_stats=self.ret_stats,
                     ret_std_out=buf.ret_std[t:t + 1] if self.ret_stats is not None else None)
            self.t_global += 1
        self.collects += 1
        if pool is not None:
            # per group: the learner's reward summed over the rollout and the episodes finished, summed over the group's
            # contiguous rows (no atomics: the same bits on every run), one copy to the host
            per_row = torch.stack([buf.rew64.sum(0), buf.done.sum(0, dtype=torch.float64)])
            rew, eps = torch.stack([per_row[:, lo:e].sum(1) for lo, e in zip([0] + ends, ends)], 1).tolist()
            rows = np.diff([0] + ends)
            self.opponent_stats = [{"snapshot_id": pool.ids[s], "rows": int(r), "mean_reward": rw / (int(r) * self.T),
                                    "episodes_finished": int(ep)} for s, r, rw, ep in zip(slots, rows, rew, eps)]
        # The reference raises where an element set is circular / parabolic (satellite_function.py:40-42 via :52-58); the
        # kernel flags the env (err = 1, dz = 0) and goes on. One reduced flag per collect() makes that visible.
        n_err = int(env.err.sum().item())
        if n_err:
            msg = f"{n_err} env(s) hit an element set for which the reference's danger-zone code raises (env.err); their rewards used dz = 0"
            if self.strict_errors:
                raise eng.L.SatError(msg)
            import warnings
            warnings.warn(msg)
        # observation after the last step (bootstrap value), normalised with the current statistics
        x = env.observe()
        if self.obs_stats is not None:
            x = (x - self.obs_stats.mean) / (self.obs_stats.std + 1e-8)
        buf.obs[self.T] = x.float()

    def compute_advantages(self, group=None, explained_variance=False):
        """explained_variance: also set self.explained_variance (device fp64 scalar) = 1 - Var(adv) / Var(v_target) over the
        rollout (all ranks of `group`), taken before the advantage normalisation; v_target - values == adv, so this is the
        rollout-level explained variance of the critic"""
        buf, ag = self.buf, self.agent
        T, n = self.T, self.env.n
        ag.critic_kernel.value(buf.obs.view(-1, 18), out=buf.values.view(-1))
        r32 = buf.rew64.float()
        r_scale = (1.0 / (buf.ret_std + 1e-8)).float() if self.ret_stats is not None else None
        eng.gae_time_major(r32, buf.values, buf.done, ag.gamma, ag.lamda, r_scale=r_scale, adv=buf.adv, v_target=buf.v_target)
        if explained_variance:
            m = torch.stack([eng.adv_moments(buf.adv), eng.adv_moments(buf.v_target)])      # [2][sum, sum of squares, count]
            dist = torch.distributed
            if group is not False and dist.is_available() and dist.is_initialized():
                pg = None if group in (None, True) else group
                if dist.get_world_size(pg) > 1:
                    dist.all_reduce(m, group=pg)
            var = m[:, 1] / m[:, 2] - (m[:, 0] / m[:, 2]) ** 2
            self.explained_variance = 1.0 - var[0] / var[1]
        if ag.use_adv_norm:
            eng.adv_normalize_(buf.adv, group=group)
        return buf.adv, buf.v_target

    def update(self, mini_batch_size: int, total_steps: int = 0, group=None, use_graph: bool = True, fused: bool = True,
               stats: bool = False):
        """fused: hand-written forward/backward/Adam kernels (csrc/ppo_update.cu); otherwise the PyTorch step, replayed as
        a CUDA graph when use_graph. Returns what the agent's optimize() returns: a PpoUpdateStats when stats (it then also
        reports explained_variance) or the agent's target_kl is set, else None."""
        buf, ag = self.buf, self.agent
        adv, v_target = self.compute_advantages(group, explained_variance=stats)
        B = self.T * self.env.n
        out = ag.optimize(buf.obs[:self.T].reshape(B, 18), buf.act.reshape(B, 3), buf.logp.reshape(B, 3), adv.reshape(B, 1),
                          v_target.reshape(B, 1), mini_batch_size=mini_batch_size, group=group, use_graph=use_graph, fused=fused,
                          stats=stats)
        if stats:
            out.extra["explained_variance"] = self.explained_variance
        if ag.use_lr_decay:
            ag.lr_decay(total_steps)
        if ag._dirty:
            ag.sync_kernels()
        return out


    # ---- full-run checkpoint: env SoA state, running normalisers, Philox counter, networks + optimisers
    def state_dict(self):
        """With stats_group set, every rank holds the same obs_stats / ret_stats, so the statistics of a state_dict() saved
        on any rank are valid for every rank; the "env" entry is the saving rank's shard."""
        ag = self.agent
        return {"env": self.env.state_dict(), "t_global": self.t_global, "seed": self.seed,
                "obs_stats": self.obs_stats.state_dict() if self.obs_stats is not None else None,
                "ret_stats": self.ret_stats.state_dict() if self.ret_stats is not None else None,
                "actor": ag.actor.state_dict(), "critic": ag.critic.state_dict(),
                "opt_actor": ag.optimizer_actor.state_dict(), "opt_critic": ag.optimizer_critic.state_dict(),
                "fused_adam": [n.state_dict() for n in ag._fused["nets"]] if ag._fused is not None else None,
                "opponent_actor": self.opponent.actor.state_dict(), "collects": self.collects,
                "opponent_pool": self.opponent_pool.state_dict() if self.opponent_pool is not None else None}

    def load_state_dict(self, sd):
        ag = self.agent
        self.env.load_state_dict(sd["env"])
        self.t_global, self.seed = int(sd["t_global"]), int(sd["seed"])
        if self.obs_stats is not None and sd["obs_stats"] is not None:
            self.obs_stats.load_state_dict(sd["obs_stats"])
        if self.ret_stats is not None and sd["ret_stats"] is not None:
            self.ret_stats.load_state_dict(sd["ret_stats"])
        ag.actor.load_state_dict(sd["actor"]); ag.critic.load_state_dict(sd["critic"])
        ag.optimizer_actor.load_state_dict(sd["opt_actor"]); ag.optimizer_critic.load_state_dict(sd["opt_critic"])
        self.opponent.actor.load_state_dict(sd["opponent_actor"])
        self.collects = int(sd.get("collects", 0))
        if self.opponent_pool is not None and sd.get("opponent_pool") is not None:
            self.opponent_pool.load_state_dict(sd["opponent_pool"])
        if sd.get("fused_adam") is not None:
            for n, st in zip(ag._fused_for(1)["nets"], sd["fused_adam"]):
                n.load_state_dict(st)
        ag.sync_kernels(); self.opponent.sync_kernels()
        return self


class SelfPlay:
    """Alternating pursuer / evader training on one device-resident env batch: the batched counterpart of CPPO_main.py's
    `Sign == 0` branch (train_pursuer_network with reset(0), :94-161, then train_evader_network with reset(1), :163-230).
    The upstream evader trainer updates the *pursuer* agent with the evader's buffer (CPPO_main.py:215); here the evader
    learns from its own rollouts, which is the evident intent.

    opponent_pool=P: each role keeps a pool of up to P snapshots of its actor (engine.OpponentPool), seeded with its initial
    actor; the end of a phase adds the learner's actor to its role's pool, and each trainer plays the other role's pool
    (VectorTrainer opponent_pool), so a learner faces a mixture of the opponent's past snapshots. Each record then carries
    "opponents": the trainer's opponent_stats."""

    def __init__(self, env: eng.EnvBatch, pursuer, evader, T: int, mini_batch_size: int, rank: int = 0, seed: int = 0,
                 opponent_pool: int | None = None, **kw):
        self.env, self.mb = env, mini_batch_size
        self.pools = None
        if opponent_pool:
            self.pools = {}
            for flag, ag in ((0, pursuer), (1, evader)):
                if ag._dirty:
                    ag.sync_kernels()
                k = ag.actor_kernel
                self.pools[flag] = eng.OpponentPool(int(opponent_pool), bool(k.use_tanh), k.max_action, k.device)
                self.pools[flag].add(k)
        p0, p1 = (self.pools[0], self.pools[1]) if self.pools else (None, None)
        self.trainers = {0: VectorTrainer(env, pursuer, evader, T, rank=rank, seed=seed, opponent_pool=p1, **kw),
                         1: VectorTrainer(env, evader, pursuer, T, rank=rank, seed=seed + 1, opponent_pool=p0, **kw)}

    def run_phase(self, flag: int, iterations: int, group=None, use_graph: bool = True, fused: bool = True, callback=None,
                  stats: bool = False):
        """stats: each iteration's record also carries the update's training diagnostics (PpoUpdateStats.as_dict keys and
        explained_variance)"""
        env, tr = self.env, self.trainers[flag]
        env.reset(flag=flag)                                   # reset(Flag) for every env; fuel / dis / dz persist (Q2)
        tr.learner_is_pursuer = flag == 0
        out = []
        for it in range(iterations):
            tr.collect()
            record = {"flag": flag, "iteration": it, "mean_reward": float(tr.buf.rew64.mean()),
                      "episodes_finished": int(tr.buf.done.sum())}
            upd = tr.update(self.mb, total_steps=it, group=group, use_graph=use_graph, fused=fused, stats=stats)
            record = dict(record, **upd.as_dict()) if stats else record
            if tr.opponent_pool is not None:
                record["opponents"] = tr.opponent_stats
            out.append(record)
            if callback is not None:
                callback(record)
        if self.pools:
            if tr.agent._dirty:
                tr.agent.sync_kernels()
            self.pools[flag].add(tr.agent.actor_kernel)          # the other role's trainer draws from this pool
        return out

    def run(self, rounds: int, iterations_per_phase: int, **kw):
        log = []
        for _ in range(rounds):
            log += self.run_phase(0, iterations_per_phase, **kw)
            log += self.run_phase(1, iterations_per_phase, **kw)
        return log


def shard_bounds(n_total: int, world: int, rank: int):
    """contiguous env shard of rank: [lo, hi)"""
    per = n_total // world
    rem = n_total % world
    lo = rank * per + min(rank, rem)
    return lo, lo + per + (1 if rank < rem else 0)
